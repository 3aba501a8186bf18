// Per-kernel C-ABI entry points (unit parity against the oracle) and the length-regulator ABI.
#include "common.cuh"

using namespace st2;

static inline int64_t align256(int64_t v) { return (v + 255) / 256 * 256; }

extern "C" {

int st2_round_durations(const float* duration, const int32_t* n_tokens, int32_t* dur, int32_t* total_frames,
                        int32_t B, int32_t L, void* stream) {
    ST2_REQUIRE(duration && dur && total_frames && B >= 0 && L >= 0, "round_durations: bad argument");
    return launch_round_durations(duration, n_tokens, dur, total_frames, B, L, (cudaStream_t)stream);
}

int st2_smooth_durations(const float* duration, const int32_t* n_tokens, const float* noise, const float* prev_d_mean, float t,
                         float speed, float* out, float* mean_out, int32_t B, int32_t L, void* stream) {
    ST2_REQUIRE(duration && out && B >= 0 && L >= 0, "smooth_durations: bad argument");
    ST2_REQUIRE(t >= 0.f && t <= 1.f && speed > 0.f, "smooth_durations: need 0 <= t <= 1 and speed > 0 (got %g, %g)", (double)t,
                (double)speed);
    ST2_REQUIRE(noise != nullptr || t == 0.f, "smooth_durations: t > 0 needs the N(0,1) tape");
    return launch_smooth_durations(duration, n_tokens, noise, prev_d_mean, t, speed, out, mean_out, B, L, (cudaStream_t)stream);
}

int st2_smooth_durations_chained(const float* duration, const int32_t* n_tokens, const float* noise, const float* prev_d_mean0, float t,
                                 float speed, float* out, float* mean_out, int32_t B, int32_t L, void* stream) {
    ST2_REQUIRE(duration && out && B >= 0 && L >= 0, "smooth_durations_chained: bad argument");
    ST2_REQUIRE(t >= 0.f && t <= 1.f && speed > 0.f, "smooth_durations_chained: need 0 <= t <= 1 and speed > 0 (got %g, %g)",
                (double)t, (double)speed);
    ST2_REQUIRE(noise != nullptr || t == 0.f, "smooth_durations_chained: t > 0 needs the N(0,1) tape");
    return launch_smooth_durations(duration, n_tokens, noise, prev_d_mean0, t, speed, out, mean_out, B, L, (cudaStream_t)stream, 1);
}

int st2_length_regulate(const float* src, const int32_t* dur, float* out, int32_t B, int32_t C, int32_t L,
                        int32_t F, int32_t channels_last, void* stream) {
    ST2_REQUIRE(B >= 0 && C >= 0 && L >= 0 && F >= 0, "length_regulate: negative size");
    if (B == 0 || C == 0 || F == 0) return ST2_OK;
    ST2_REQUIRE(src && dur && out, "length_regulate: null tensor");
    return launch_length_regulate(src, dur, out, B, C, L, F, channels_last, (cudaStream_t)stream);
}

int st2_sinegen_phase(const float* f0, float* phase, float* frames_scratch, int32_t B, int32_t L2,
                      int32_t upsample_scale, void* stream) {
    ST2_REQUIRE(f0 && phase && frames_scratch && B > 0 && L2 > 0 && upsample_scale > 0, "sinegen_phase: bad argument");
    int e = launch_sinegen_frames(f0, frames_scratch, B, L2, upsample_scale, (cudaStream_t)stream);
    if (e != ST2_OK) return e;
    return launch_sinegen_phase(frames_scratch, phase, B, L2, upsample_scale, (cudaStream_t)stream);
}

int st2_har_source(const float* f0, const float* noise, uint64_t seed, const float* lin_w, const float* lin_b,
                   float* har, float* frames_scratch, int32_t B, int32_t L2, int32_t upsample_scale, void* stream) {
    ST2_REQUIRE(f0 && lin_w && lin_b && har && frames_scratch && B > 0 && L2 > 0 && upsample_scale > 0,
                "har_source: bad argument");
    int e = launch_sinegen_frames(f0, frames_scratch, B, L2, upsample_scale, (cudaStream_t)stream);
    if (e != ST2_OK) return e;
    return launch_har_source(f0, frames_scratch, noise, seed, nullptr, lin_w, lin_b, har, B, L2, upsample_scale,
                             (cudaStream_t)stream);
}

// generator.noise_convs[i] + the AdaIN coefficients of its output, as the decoder runs them (decoder.cu, Exec::resblock1)
static int64_t noise_conv_offsets(int B, int Tout, int C, int k, int stride, int64_t off[2]) {
    int64_t o = 0;
    off[0] = o; o += align256((int64_t)k * C * sizeof(float));                                  // packed weight [k][C]
    off[1] = o; o += align256((int64_t)B * noise_conv_parts(Tout, stride) * C * 8);             // float2 tile partials
    return o;
}

int64_t st2_noise_conv_scratch_bytes(int32_t B, int32_t Tout, int32_t C, int32_t k, int32_t stride) {
    if (B <= 0 || Tout <= 0 || C <= 0 || k <= 0 || stride <= 0) return ST2_ERR_INVALID;
    int64_t off[2];
    return noise_conv_offsets(B, Tout, C, k, stride, off);
}

int st2_noise_conv(const float* har, const float* w, const float* bias, void* y, const float* h, float* coef, void* scratch,
                   int32_t B, int32_t S, int32_t Tout, int32_t C, int32_t k, int32_t stride, int32_t pad, int32_t y16,
                   void* stream) {
    ST2_REQUIRE(har && w && bias && y && scratch && B > 0 && S > 0 && C > 0 && k > 0 && stride > 0 && pad >= 0,
                "noise_conv: bad argument");
    ST2_REQUIRE(Tout == (S + 2 * pad - k) / stride + 1 && Tout > 0, "noise_conv: Tout=%d does not match S=%d k=%d stride=%d pad=%d",
                Tout, S, k, stride, pad);
    ST2_REQUIRE((h == nullptr) == (coef == nullptr), "noise_conv: h and coef go together");
    cudaStream_t st = (cudaStream_t)stream;
    int64_t off[2];
    noise_conv_offsets(B, Tout, C, k, stride, off);
    float* wp = (float*)((char*)scratch + off[0]);
    void* parts = (char*)scratch + off[1];
    int e = launch_fold_pack(nullptr, w, wp, C, 1, k, 0, st);
    if (e == ST2_OK) e = launch_noise_conv(har, wp, bias, (float*)y, parts, B, S, Tout, C, k, stride, pad, st, y16 ? 1 : 0);
    // the partials are of y - bias; the fp16 y is stored without the bias
    if (e == ST2_OK && h != nullptr)
        e = launch_adain_coef_f2(parts, noise_conv_parts(Tout, stride), h, 2 * C, 0, coef, B, Tout, C, C, st, y16 ? bias : nullptr,
                                 bias);
    return e;
}

int st2_post_hifigan(const void* x, int32_t ld_x, const float* alpha, const float* w, const float* bias, float* out,
                     float* w_scratch, int32_t B, int32_t S, int32_t C, int32_t fast, int32_t x16, void* stream) {
    ST2_REQUIRE(x && alpha && w && bias && out && w_scratch && B > 0 && S > 0 && C > 0 && ld_x >= C, "post_hifigan: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    int e = launch_fold_pack(nullptr, w, w_scratch, 1, C, 7, 0, st);
    if (e != ST2_OK) return e;
    return launch_post_hifigan((const float*)x, ld_x, alpha, w_scratch, bias, out, B, S, C, fast ? 1 : 0, st, x16 ? 1 : 0);
}

int st2_style_fc(const float* s, const float* W, const float* bias, float* h, int32_t B, int32_t R, int32_t K, void* stream) {
    ST2_REQUIRE(s && W && bias && h && B > 0 && R > 0 && K > 0, "style_fc: bad argument");
    return launch_style_fc(s, W, bias, h, B, R, K, (cudaStream_t)stream);
}

int64_t st2_adain_scratch_bytes(int32_t B, int32_t T, int32_t C) {
    if (B <= 0 || T <= 0 || C <= 0) return ST2_ERR_INVALID;
    const int Cpad = (C + 3) / 4 * 4;
    return align256(adain_scratch_bytes(B, T, C)) + align256((int64_t)B * 2 * Cpad * sizeof(float));
}

int st2_adain_act(const float* x, int32_t ld_x, const float* h, int32_t ld_h, const float* alpha, int32_t act,
                  float slope, void* y, int32_t ld_y, int32_t out_dtype, int32_t B, int32_t T, int32_t C,
                  void* scratch, void* stream) {
    ST2_REQUIRE(x && y && scratch && B > 0 && T > 0 && C > 0, "adain_act: bad argument");
    ST2_REQUIRE(C % 4 == 0, "adain_act: C=%d must be a multiple of 4", C);
    cudaStream_t st = (cudaStream_t)stream;
    float* coef = (float*)((char*)scratch + align256(adain_scratch_bytes(B, T, C)));
    int e = ST2_OK;
    if (h != nullptr) {
        e = launch_in_stats(x, ld_x, B, T, C, scratch, st);
        if (e != ST2_OK) return e;
    }
    e = launch_adain_coef(scratch, h, ld_h, 0, coef, B, T, C, C, st);
    if (e != ST2_OK) return e;
    return launch_affine_act(x, ld_x, coef, alpha, act, slope, y, ld_y, out_dtype, B, T, C, st);
}

int64_t st2_conv1d_scratch_bytes(int32_t B, int32_t Tin, int32_t Cin, int32_t Cout, int32_t k, int32_t precision) {
    if (B <= 0 || Tin <= 0 || Cin <= 0 || Cout <= 0 || k <= 0) return ST2_ERR_INVALID;
    int64_t bytes = align256((int64_t)k * Cin * Cout * sizeof(float));
    if (precision != ST2_PREC_FP32) {
        const int cin_pad = (Cin + 63) / 64 * 64, cout_pad = (Cout + 15) / 16 * 16;
        bytes += align256((int64_t)k * cin_pad * cout_pad * 2);
        bytes += align256((int64_t)B * Tin * cin_pad * 2);       // 16-bit copy of x
        bytes += align256((int64_t)B * 2 * cin_pad * sizeof(float));
    }
    return bytes;
}

int st2_conv1d(const float* x, const float* w, const float* bias, float* y, void* scratch, int32_t B, int32_t Tin,
               int32_t Cin, int32_t Cout, int32_t k, int32_t stride, int32_t padding, int32_t dilation,
               int32_t output_padding, int32_t transposed, int32_t precision, void* stream) {
    ST2_REQUIRE(x && w && y && scratch && B > 0 && Tin > 0 && Cin > 0 && Cout > 0 && k > 0 && stride > 0 && dilation > 0,
                "conv1d: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    float* wp = (float*)scratch;
    const int d0 = transposed ? Cin : Cout, d1 = transposed ? Cout : Cin;
    int e = launch_fold_pack(nullptr, w, wp, d0, d1, k, transposed ? 1 : 0, st);
    if (e != ST2_OK) return e;
    ConvArgs a;
    memset(&a, 0, sizeof(a));
    a.B = B; a.Cin = Cin; a.Cout = Cout; a.Tin = Tin;
    a.w = wp; a.bias = bias; a.y = y; a.ld_y = Cout; a.scale = 1.f;
    if (!transposed) {
        a.Tout = (Tin + 2 * padding - dilation * (k - 1) - 1) / stride + 1;
        a.M = a.Tout; a.ntaps = k; a.tap_step = dilation; a.in_off = -padding; a.in_stride = stride;
        a.phases = 1; a.w_step = 1; a.out_stride = 1; a.out_pad = 0;
    } else {
        ST2_REQUIRE(k % stride == 0 && dilation == 1, "conv1d: transposed needs k %% stride == 0 and dilation 1");
        a.Tout = (Tin - 1) * stride - 2 * padding + (k - 1) + output_padding + 1;
        a.ntaps = k / stride; a.tap_step = -1; a.in_off = 0; a.in_stride = 1;
        a.phases = stride; a.w_step = stride; a.out_stride = stride; a.out_pad = padding;
        a.M = (a.Tout - 1 + padding) / stride + 1;
    }
    ST2_REQUIRE(a.Tout > 0, "conv1d: empty output");
    if (precision == ST2_PREC_FP32) {
        a.x = x; a.ld_x = Cin;
        return launch_conv_simt(a, st);
    }
    const int dt = precision == ST2_PREC_BF16 ? DT_BF16 : DT_F16;
    const int cin_pad = (Cin + 63) / 64 * 64, cout_pad = (Cout + 15) / 16 * 16;
    char* p = (char*)scratch + align256((int64_t)k * Cin * Cout * sizeof(float));
    void* w16 = p;
    p += align256((int64_t)k * cin_pad * cout_pad * 2);
    void* x16 = p;
    p += align256((int64_t)B * Tin * cin_pad * 2);
    float* coef = (float*)p;
    e = launch_pack_w16(wp, w16, k, Cin, Cout, cin_pad, cout_pad, dt, st);
    if (e != ST2_OK) return e;
    ST2_REQUIRE(Cin % 4 == 0, "conv1d: tensor-core unit path needs Cin %% 4 == 0");
    // 16-bit, channel-padded copy of x (identity affine)
    ST2_CUDA_CHECK(cudaMemsetAsync(x16, 0, (size_t)B * Tin * cin_pad * 2, st));
    e = launch_adain_coef(nullptr, nullptr, 0, 0, coef, B, Tin, Cin, Cin, st);
    if (e != ST2_OK) return e;
    e = launch_affine_act(x, Cin, coef, nullptr, ACT_NONE, 0.f, x16, cin_pad, dt, B, Tin, Cin, st);
    if (e != ST2_OK) return e;
    a.x16 = x16; a.ld_x16 = cin_pad; a.w16 = w16; a.w16_cin_pad = cin_pad; a.w16_cout_pad = cout_pad; a.fmt16 = dt;
    return launch_conv_tc(a, st);
}

// One fused half-step of AdaINResBlock1 (hifigan.py:67-73) through the tensor-core fused kernels:
//   y = (conv1d(act(AdaIN(x; h)), w) + bias + res (+ y_old)) * scale,   coef_next = AdaIN coefficients of y for style h_next
static int64_t fused_unit_offsets(int B, int T, int Cin, int Cout, int k, int64_t off[6]) {
    const int cin_pad = (Cin + 63) / 64 * 64, cout_pad = (Cout + 31) / 32 * 32;
    int64_t o = 0;
    off[0] = o; o += align256((int64_t)k * Cin * Cout * sizeof(float));          // packed fp32 weight
    off[1] = o; o += align256((int64_t)k * cin_pad * cout_pad * 2);              // 16-bit weight
    off[2] = o; o += align256(adain_scratch_bytes(B, T, Cin));                   // input statistics
    off[3] = o; o += align256((int64_t)B * 2 * cin_pad * sizeof(float));         // input coefficients
    off[4] = o; o += align256((int64_t)B * (cdiv(T, 128) * 4) * Cout * 8);       // output partials
    off[5] = o;
    return o;
}

int64_t st2_adain_conv1d_fused_scratch_bytes(int32_t B, int32_t T, int32_t Cin, int32_t Cout, int32_t k) {
    if (B <= 0 || T <= 0 || Cin <= 0 || Cout <= 0 || k <= 0) return ST2_ERR_INVALID;
    int64_t off[6];
    return fused_unit_offsets(B, T, Cin, Cout, k, off);
}

int st2_adain_conv1d_fused(const float* x, const float* h, const float* alpha, int32_t act, float slope, const float* w,
                           const float* bias, const float* res, float* y, const float* h_next, float* coef_next,
                           void* scratch, int32_t B, int32_t T, int32_t Cin, int32_t Cout, int32_t k, int32_t padding,
                           int32_t dilation, float scale, int32_t accumulate, int32_t precision, void* stream) {
    ST2_REQUIRE(x && w && y && scratch && B > 0 && T > 0 && Cin > 0 && Cout > 0 && k > 0 && dilation > 0,
                "adain_conv1d_fused: bad argument");
    ST2_REQUIRE(precision == ST2_PREC_BF16 || precision == ST2_PREC_FP16, "adain_conv1d_fused: 16-bit precisions only");
    ST2_REQUIRE(2 * padding == dilation * (k - 1), "adain_conv1d_fused: length-preserving convolutions only");
    ST2_REQUIRE((h_next == nullptr) == (coef_next == nullptr), "adain_conv1d_fused: h_next and coef_next go together");
    cudaStream_t st = (cudaStream_t)stream;
    int64_t off[6];
    fused_unit_offsets(B, T, Cin, Cout, k, off);
    char* base = (char*)scratch;
    float* wp = (float*)(base + off[0]);
    void* w16 = base + off[1];
    void* xstats = base + off[2];
    float* coef = (float*)(base + off[3]);
    void* parts = base + off[4];
    const int dt = precision == ST2_PREC_BF16 ? DT_BF16 : DT_F16;
    const int cin_pad = (Cin + 63) / 64 * 64, cout_pad = (Cout + 31) / 32 * 32;
    int e = launch_fold_pack(nullptr, w, wp, Cout, Cin, k, 0, st);
    if (e != ST2_OK) return e;
    e = launch_pack_w16(wp, w16, k, Cin, Cout, cin_pad, cout_pad, dt, st);
    if (e != ST2_OK) return e;
    if (h != nullptr) {
        e = launch_in_stats(x, Cin, B, T, Cin, xstats, st);
        if (e != ST2_OK) return e;
    }
    e = launch_adain_coef(xstats, h, 2 * Cin, 0, coef, B, T, Cin, Cin, st);
    if (e != ST2_OK) return e;
    ConvArgs a;
    memset(&a, 0, sizeof(a));
    a.B = B; a.Cin = Cin; a.Cout = Cout; a.Tin = T; a.Tout = T; a.M = T;
    a.x = x; a.ld_x = Cin; a.w = wp; a.w16 = w16; a.w16_cin_pad = cin_pad; a.w16_cout_pad = cout_pad; a.fmt16 = dt;
    a.bias = bias; a.res = res; a.ld_res = Cout; a.y = y; a.ld_y = Cout;
    a.ntaps = k; a.tap_step = dilation; a.in_off = -padding; a.in_stride = 1;
    a.phases = 1; a.w_step = 1; a.out_stride = 1; a.out_pad = 0;
    a.scale = scale; a.accumulate = accumulate;
    ST2_REQUIRE(conv_fused_supported(a), "adain_conv1d_fused: geometry not supported by the fused kernels");
    e = launch_conv_fused(a, coef, Cin, act, slope, alpha, h_next ? parts : nullptr, st);
    if (e != ST2_OK) return e;
    if (h_next != nullptr) e = launch_adain_coef_f2(parts, fused_stats_parts(a), h_next, 2 * Cout, 0, coef_next, B, T, Cout, Cout, st);
    return e;
}

// st2_adain_conv1d_fused with the fp16 storage types of the decoder's resblocks (program.cuh resblock1): x, res, old are given
// as fp32 tensors and stored as fp16 first when their flag says so; y is written as fp16 and widened when y16.  A separate
// accumulate source `old` (fp32 or fp16) replaces the old values in y; with old_in_y it is first stored into the fp16 y buffer
// and the conv accumulates in place, as the middle resblock of a stage updates the fp16 stage sum.
static int64_t fused_ex_offsets(int B, int T, int Cin, int Cout, int k, int64_t off[11]) {
    int64_t o = fused_unit_offsets(B, T, Cin, Cout, k, off);
    off[6] = o; o += align256((int64_t)B * T * Cin * 2);                         // x as fp16
    off[7] = o; o += align256((int64_t)B * T * Cout * 2);                        // res as fp16
    off[8] = o; o += align256((int64_t)B * T * Cout * 2);                        // old as fp16
    off[9] = o; o += align256((int64_t)B * T * Cout * 2);                        // y as fp16
    off[10] = o;
    return o;
}

int64_t st2_adain_conv1d_fused_ex_scratch_bytes(int32_t B, int32_t T, int32_t Cin, int32_t Cout, int32_t k) {
    if (B <= 0 || T <= 0 || Cin <= 0 || Cout <= 0 || k <= 0) return ST2_ERR_INVALID;
    int64_t off[11];
    return fused_ex_offsets(B, T, Cin, Cout, k, off);
}

int st2_adain_conv1d_fused_ex(const float* x, const float* h, const float* alpha, int32_t act, float slope, const float* w,
                              const float* bias, const float* res, const float* old, float* y, const float* h_next,
                              float* coef_next, void* scratch, int32_t B, int32_t T, int32_t Cin, int32_t Cout, int32_t k,
                              int32_t padding, int32_t dilation, float scale, int32_t accumulate, int32_t x16, int32_t res16,
                              int32_t old16, int32_t y16, int32_t old_in_y, int32_t precision, void* stream) {
    ST2_REQUIRE(x && w && y && scratch && B > 0 && T > 0 && Cin > 0 && Cout > 0 && k > 0 && dilation > 0,
                "adain_conv1d_fused_ex: bad argument");
    ST2_REQUIRE(precision == ST2_PREC_BF16 || precision == ST2_PREC_FP16, "adain_conv1d_fused_ex: 16-bit precisions only");
    ST2_REQUIRE(2 * padding == dilation * (k - 1), "adain_conv1d_fused_ex: length-preserving convolutions only");
    ST2_REQUIRE((h_next == nullptr) == (coef_next == nullptr), "adain_conv1d_fused_ex: h_next and coef_next go together");
    ST2_REQUIRE(!res16 || res != nullptr, "adain_conv1d_fused_ex: res16 needs a residual");
    ST2_REQUIRE(old == nullptr || accumulate, "adain_conv1d_fused_ex: a separate accumulate source needs accumulate");
    ST2_REQUIRE(!old16 || old != nullptr, "adain_conv1d_fused_ex: old16 needs old values");
    ST2_REQUIRE(!old_in_y || (old16 && y16), "adain_conv1d_fused_ex: old_in_y accumulates in place on an fp16 y (old16, y16)");
    cudaStream_t st = (cudaStream_t)stream;
    int64_t off[11];
    fused_ex_offsets(B, T, Cin, Cout, k, off);
    char* base = (char*)scratch;
    float* wp = (float*)(base + off[0]);
    void* w16 = base + off[1];
    void* xstats = base + off[2];
    float* coef = (float*)(base + off[3]);
    void* parts = base + off[4];
    void* x16b = base + off[6];
    void* r16b = base + off[7];
    void* o16b = base + off[8];
    void* y16b = base + off[9];
    const int dt = precision == ST2_PREC_BF16 ? DT_BF16 : DT_F16;
    const int cin_pad = (Cin + 63) / 64 * 64, cout_pad = (Cout + 31) / 32 * 32;
    const int64_t n_in = (int64_t)B * T * Cin, n_out = (int64_t)B * T * Cout;
    int e = launch_fold_pack(nullptr, w, wp, Cout, Cin, k, 0, st);
    if (e == ST2_OK) e = launch_pack_w16(wp, w16, k, Cin, Cout, cin_pad, cout_pad, dt, st);
    if (e == ST2_OK && h != nullptr) e = launch_in_stats(x, Cin, B, T, Cin, xstats, st);
    if (e == ST2_OK) e = launch_adain_coef(xstats, h, 2 * Cin, 0, coef, B, T, Cin, Cin, st);
    if (e == ST2_OK && x16) e = launch_cast16(x, x16b, n_in, DT_F16, st);
    if (e == ST2_OK && res16) e = launch_cast16(res, r16b, n_out, DT_F16, st);
    if (e == ST2_OK && old16) e = launch_cast16(old, old_in_y ? y16b : o16b, n_out, DT_F16, st);
    if (e != ST2_OK) return e;
    ConvArgs a;
    memset(&a, 0, sizeof(a));
    a.B = B; a.Cin = Cin; a.Cout = Cout; a.Tin = T; a.Tout = T; a.M = T;
    a.x = x16 ? (const float*)x16b : x; a.ld_x = Cin; a.x16in = x16 ? 1 : 0;
    a.w = wp; a.w16 = w16; a.w16_cin_pad = cin_pad; a.w16_cout_pad = cout_pad; a.fmt16 = dt;
    a.bias = bias; a.res = res16 ? (const float*)r16b : res; a.ld_res = Cout; a.res16 = res16 ? 1 : 0;
    a.y = y16 ? (float*)y16b : y; a.ld_y = Cout; a.y16out = y16 ? 1 : 0;
    a.ntaps = k; a.tap_step = dilation; a.in_off = -padding; a.in_stride = 1;
    a.phases = 1; a.w_step = 1; a.out_stride = 1; a.out_pad = 0;
    a.scale = scale; a.accumulate = accumulate ? 1 : 0;
    if (old != nullptr) {
        a.acc_src = old16 ? (old_in_y ? y16b : o16b) : (const void*)old;
        a.acc16 = old16 ? 1 : 0;
    }
    ST2_REQUIRE(conv_fused_supported(a), "adain_conv1d_fused_ex: geometry not supported by the fused kernels");
    ST2_REQUIRE(!(x16 || res16 || old16 || y16) || conv_pipe_supported(a),
                "adain_conv1d_fused_ex: these fp16 storage types need the TMA pipeline kernel, which cannot run this geometry");
    e = launch_conv_fused(a, coef, Cin, act, slope, alpha, h_next ? parts : nullptr, st);
    if (e == ST2_OK && y16) e = launch_half_to_float(y16b, y, n_out, st);
    if (e == ST2_OK && h_next != nullptr)
        e = launch_adain_coef_f2(parts, fused_stats_parts(a), h_next, 2 * Cout, 0, coef_next, B, T, Cout, Cout, st);
    return e;
}

// The same half-step on the row-per-thread kernel (conv_row.cu) with the storage types of the 16-bit decoder paths: x, res
// and old are given as fp32 tensors and are stored as fp16 first when the x16 flag says so / always (res, old); y is written as fp16
// and widened when y16.  C = Cin = Cout in {32, 64}, Snake only.
static int64_t row_unit_offsets(int B, int T, int C, int k, int64_t off[10]) {
    int64_t o = 0;
    off[0] = o; o += align256((int64_t)k * C * C * sizeof(float));               // packed fp32 weight
    off[1] = o; o += align256((int64_t)k * 64 * C * 2);                          // 16-bit weight
    off[2] = o; o += align256(adain_scratch_bytes(B, T, C));                     // input statistics
    off[3] = o; o += align256((int64_t)B * 2 * C * sizeof(float));               // input coefficients
    off[4] = o; o += align256(conv_row_stats_bytes(B, T, C));                    // output partials
    off[5] = o; o += align256((int64_t)B * T * C * 2);                           // x as fp16
    off[6] = o; o += align256((int64_t)B * T * C * 2);                           // res as fp16
    off[7] = o; o += align256((int64_t)B * T * C * 2);                           // old as fp16
    off[8] = o; o += align256((int64_t)B * T * C * 2);                           // y as fp16
    off[9] = o;
    return o;
}

int64_t st2_adain_conv1d_row_scratch_bytes(int32_t B, int32_t T, int32_t C, int32_t k) {
    if (B <= 0 || T <= 0 || !(C == 32 || C == 64) || k <= 0) return ST2_ERR_INVALID;
    int64_t off[10];
    return row_unit_offsets(B, T, C, k, off);
}

int st2_adain_conv1d_row(const float* x, const float* h, const float* alpha, const float* w, const float* bias,
                         const float* res, const float* old, float* y, const float* h_next, float* coef_next, void* scratch,
                         int32_t B, int32_t T, int32_t C, int32_t k, int32_t padding, int32_t dilation, float scale,
                         int32_t precision, int32_t x16, int32_t y16, void* stream) {
    ST2_REQUIRE(x && h && alpha && w && y && scratch && B > 0 && T > 0 && (C == 32 || C == 64) && k > 0 && dilation > 0,
                "adain_conv1d_row: bad argument");
    ST2_REQUIRE(precision == ST2_PREC_BF16 || precision == ST2_PREC_FP16, "adain_conv1d_row: 16-bit precisions only");
    ST2_REQUIRE(2 * padding == dilation * (k - 1), "adain_conv1d_row: length-preserving convolutions only");
    ST2_REQUIRE((h_next == nullptr) == (coef_next == nullptr), "adain_conv1d_row: h_next and coef_next go together");
    ST2_REQUIRE(old == nullptr || res != nullptr, "adain_conv1d_row: old values need a residual");
    cudaStream_t st = (cudaStream_t)stream;
    int64_t off[10];
    row_unit_offsets(B, T, C, k, off);
    char* base = (char*)scratch;
    float* wp = (float*)(base + off[0]);
    void* w16 = base + off[1];
    void* xstats = base + off[2];
    float* coef = (float*)(base + off[3]);
    void* parts = base + off[4];
    void* x16b = base + off[5];
    void* r16b = base + off[6];
    void* o16b = base + off[7];
    void* y16b = base + off[8];
    const int dt = precision == ST2_PREC_BF16 ? DT_BF16 : DT_F16;
    const int64_t n = (int64_t)B * T * C;
    int e = launch_fold_pack(nullptr, w, wp, C, C, k, 0, st);
    if (e != ST2_OK) return e;
    e = launch_pack_w16(wp, w16, k, C, C, 64, C, dt, st);
    if (e != ST2_OK) return e;
    e = launch_in_stats(x, C, B, T, C, xstats, st);
    if (e != ST2_OK) return e;
    e = launch_adain_coef(xstats, h, 2 * C, 0, coef, B, T, C, C, st);
    if (e != ST2_OK) return e;
    if (x16) { e = launch_cast16(x, x16b, n, DT_F16, st); if (e != ST2_OK) return e; }
    if (res) { e = launch_cast16(res, r16b, n, DT_F16, st); if (e != ST2_OK) return e; }
    if (old) { e = launch_cast16(old, o16b, n, DT_F16, st); if (e != ST2_OK) return e; }
    ConvArgs a;
    memset(&a, 0, sizeof(a));
    a.B = B; a.Cin = C; a.Cout = C; a.Tin = T; a.Tout = T; a.M = T;
    a.x = x16 ? (const float*)x16b : x; a.ld_x = C; a.x16in = x16 ? 1 : 0;
    a.w = wp; a.w16 = w16; a.w16_cin_pad = 64; a.w16_cout_pad = C; a.fmt16 = dt;
    a.bias = bias;
    if (res) { a.res = (const float*)r16b; a.ld_res = C; a.res16 = 1; }
    if (old) { a.accumulate = 1; a.acc_src = o16b; a.acc16 = 1; }
    a.y = y16 ? (float*)y16b : y; a.ld_y = C; a.y16out = y16 ? 1 : 0;
    a.ntaps = k; a.tap_step = dilation; a.in_off = -padding; a.in_stride = 1;
    a.phases = 1; a.w_step = 1; a.out_stride = 1; a.out_pad = 0;
    a.scale = scale;
    ST2_REQUIRE(conv_row_can_launch(a), "adain_conv1d_row: geometry not supported by conv_row");
    RowStatsDesc rd;
    e = launch_conv_row(a, coef, C, ACT_SNAKE, alpha, h_next ? parts : nullptr, &rd, st);
    if (e != ST2_OK) return e;
    if (y16) { e = launch_half_to_float(y16b, y, n, st); if (e != ST2_OK) return e; }
    if (h_next != nullptr) e = launch_adain_coef_row(parts, rd, h_next, 2 * C, 0, coef_next, B, T, C, C, st);
    return e;
}

// Two chained half-steps on conv_row.cu as one iteration of AdaINResBlock1 runs them in the decoder: the second launch reads the
// first one's fp16 output and, when its coefficient table fits, computes that output's AdaIN coefficients itself from the
// first launch's statistics partials (RowCoefSrc) instead of from a coefficient launch in between.
static int64_t row_pair_offsets(int B, int T, int C, int k1, int k2, int64_t off[13]) {
    int64_t o = 0;
    off[0] = o; o += align256((int64_t)k1 * C * C * sizeof(float));              // packed fp32 weights of step 1
    off[1] = o; o += align256((int64_t)k1 * 64 * C * 2);                         // 16-bit weights of step 1
    off[2] = o; o += align256((int64_t)k2 * C * C * sizeof(float));              // step 2
    off[3] = o; o += align256((int64_t)k2 * 64 * C * 2);
    off[4] = o; o += align256(adain_scratch_bytes(B, T, C));                     // statistics of x
    off[5] = o; o += align256((int64_t)B * 2 * C * sizeof(float));               // coefficients of x
    off[6] = o; o += align256((int64_t)B * 2 * C * sizeof(float));               // coefficients of y1 (coefficient-kernel path)
    off[7] = o; o += align256(conv_row_stats_bytes(B, T, C));                    // partials of y1
    off[8] = o; o += align256(conv_row_stats_bytes(B, T, C));                    // partials of y2
    off[9] = o; o += align256((int64_t)B * T * C * 2);                           // x as fp16
    off[10] = o; o += align256((int64_t)B * T * C * 2);                          // y1 as fp16
    off[11] = o; o += align256((int64_t)B * T * C * 2);                          // y2 as fp16
    off[12] = o;
    return o;
}

int64_t st2_adain_conv1d_row_pair_scratch_bytes(int32_t B, int32_t T, int32_t C, int32_t k1, int32_t k2) {
    if (B <= 0 || T <= 0 || !(C == 32 || C == 64) || k1 <= 0 || k2 <= 0) return ST2_ERR_INVALID;
    int64_t off[13];
    return row_pair_offsets(B, T, C, k1, k2, off);
}

int st2_adain_conv1d_row_pair(const float* x, const float* h1, const float* alpha1, const float* w1, const float* bias1,
                              const float* h2, const float* alpha2, const float* w2, const float* bias2, float* y1, float* y2,
                              const float* h_next, float* coef_next, int32_t* inline_coef, void* scratch, int32_t B, int32_t T,
                              int32_t C, int32_t k1, int32_t dil1, int32_t k2, int32_t dil2, int32_t precision, void* stream) {
    ST2_REQUIRE(x && h1 && alpha1 && w1 && h2 && alpha2 && w2 && y1 && y2 && scratch && B > 0 && T > 0 && (C == 32 || C == 64) &&
                    k1 > 0 && k2 > 0 && dil1 > 0 && dil2 > 0,
                "adain_conv1d_row_pair: bad argument");
    ST2_REQUIRE(precision == ST2_PREC_BF16 || precision == ST2_PREC_FP16, "adain_conv1d_row_pair: 16-bit precisions only");
    ST2_REQUIRE(dil1 * (k1 - 1) % 2 == 0 && dil2 * (k2 - 1) % 2 == 0, "adain_conv1d_row_pair: length-preserving convolutions only");
    ST2_REQUIRE((h_next == nullptr) == (coef_next == nullptr), "adain_conv1d_row_pair: h_next and coef_next go together");
    cudaStream_t st = (cudaStream_t)stream;
    int64_t off[13];
    row_pair_offsets(B, T, C, k1, k2, off);
    char* base = (char*)scratch;
    float* wp1 = (float*)(base + off[0]);
    void* w16_1 = base + off[1];
    float* wp2 = (float*)(base + off[2]);
    void* w16_2 = base + off[3];
    void* xstats = base + off[4];
    float* coef1 = (float*)(base + off[5]);
    float* coef2 = (float*)(base + off[6]);
    void* parts1 = base + off[7];
    void* parts2 = base + off[8];
    void* x16b = base + off[9];
    void* y1_16 = base + off[10];
    void* y2_16 = base + off[11];
    const int dt = precision == ST2_PREC_BF16 ? DT_BF16 : DT_F16;
    const int64_t n = (int64_t)B * T * C;
    int e = launch_fold_pack(nullptr, w1, wp1, C, C, k1, 0, st);
    if (e == ST2_OK) e = launch_pack_w16(wp1, w16_1, k1, C, C, 64, C, dt, st);
    if (e == ST2_OK) e = launch_fold_pack(nullptr, w2, wp2, C, C, k2, 0, st);
    if (e == ST2_OK) e = launch_pack_w16(wp2, w16_2, k2, C, C, 64, C, dt, st);
    if (e == ST2_OK) e = launch_in_stats(x, C, B, T, C, xstats, st);
    if (e == ST2_OK) e = launch_adain_coef(xstats, h1, 2 * C, 0, coef1, B, T, C, C, st);
    if (e == ST2_OK) e = launch_cast16(x, x16b, n, DT_F16, st);
    if (e != ST2_OK) return e;
    ConvArgs a1;
    memset(&a1, 0, sizeof(a1));
    a1.B = B; a1.Cin = C; a1.Cout = C; a1.Tin = T; a1.Tout = T; a1.M = T;
    a1.x = (const float*)x16b; a1.ld_x = C; a1.x16in = 1;
    a1.w = wp1; a1.w16 = w16_1; a1.w16_cin_pad = 64; a1.w16_cout_pad = C; a1.fmt16 = dt;
    a1.bias = bias1;
    a1.y = (float*)y1_16; a1.ld_y = C; a1.y16out = 1;
    a1.ntaps = k1; a1.tap_step = dil1; a1.in_off = -dil1 * (k1 - 1) / 2; a1.in_stride = 1;
    a1.phases = 1; a1.w_step = 1; a1.out_stride = 1; a1.out_pad = 0;
    a1.scale = 1.f;
    ConvArgs a2 = a1;                              // y2 = conv(snake(AdaIN(y1))) + bias2 + x
    a2.x = (const float*)y1_16;
    a2.w = wp2; a2.w16 = w16_2;
    a2.bias = bias2;
    a2.res = (const float*)x16b; a2.ld_res = C; a2.res16 = 1;
    a2.y = (float*)y2_16;
    a2.ntaps = k2; a2.tap_step = dil2; a2.in_off = -dil2 * (k2 - 1) / 2;
    ST2_REQUIRE(conv_row_can_launch(a1) && conv_row_can_launch(a2), "adain_conv1d_row_pair: geometry not supported by conv_row");
    RowStatsDesc rd1, rd2;
    e = launch_conv_row(a1, coef1, C, ACT_SNAKE, alpha1, parts1, &rd1, st);
    if (e != ST2_OK) return e;
    const bool inl = conv_row_inline_coef_ok(a2);
    if (inline_coef != nullptr) *inline_coef = inl ? 1 : 0;
    const RowCoefSrc src{parts1, rd1, h2, 2 * C, 0, T};
    if (!inl) {
        e = launch_adain_coef_row(parts1, rd1, h2, 2 * C, 0, coef2, B, T, C, C, st);
        if (e != ST2_OK) return e;
    }
    e = launch_conv_row(a2, coef2, C, ACT_SNAKE, alpha2, h_next ? parts2 : nullptr, &rd2, st, inl ? &src : nullptr);
    if (e == ST2_OK) e = launch_half_to_float(y1_16, y1, n, st);
    if (e == ST2_OK) e = launch_half_to_float(y2_16, y2, n, st);
    if (e == ST2_OK && h_next != nullptr) e = launch_adain_coef_row(parts2, rd2, h_next, 2 * C, 0, coef_next, B, T, C, C, st);
    return e;
}

// Generator upsampling step (hifigan.py:329-334): y = conv_transpose1d(act(x), w) + bias + res, plus the AdaIN
// coefficients of y for style h_next, through the fused tensor-core kernels.
static int64_t fused_t_offsets(int B, int Tin, int Cin, int Cout, int k, int stride, int64_t off[5]) {
    const int cin_pad = (Cin + 63) / 64 * 64, cout_pad = (Cout + 31) / 32 * 32;
    const int M = Tin + k / stride;                                                    // >= rows of any phase
    int64_t o = 0;
    off[0] = o; o += align256((int64_t)k * Cin * Cout * sizeof(float));               // packed fp32 weight
    off[1] = o; o += align256((int64_t)k * cin_pad * cout_pad * 2);                   // 16-bit weight
    off[2] = o; o += align256((int64_t)B * 2 * cin_pad * sizeof(float));              // identity coefficients
    off[3] = o; o += align256((int64_t)B * ((int64_t)stride * cdiv(M, 128) * 4) * Cout * 8);   // output partials
    off[4] = o;
    return o;
}

int64_t st2_act_conv_transpose1d_fused_scratch_bytes(int32_t B, int32_t Tin, int32_t Cin, int32_t Cout, int32_t k,
                                                     int32_t stride) {
    if (B <= 0 || Tin <= 0 || Cin <= 0 || Cout <= 0 || k <= 0 || stride <= 0) return ST2_ERR_INVALID;
    int64_t off[5];
    return fused_t_offsets(B, Tin, Cin, Cout, k, stride, off);
}

int st2_act_conv_transpose1d_fused(const float* x, const float* alpha, int32_t act, float slope, const float* w,
                                   const float* bias, const float* res, float* y, const float* h_next, float* coef_next,
                                   void* scratch, int32_t B, int32_t Tin, int32_t Cin, int32_t Cout, int32_t k,
                                   int32_t stride, int32_t padding, int32_t output_padding, int32_t precision, void* stream) {
    ST2_REQUIRE(x && w && y && scratch && B > 0 && Tin > 0 && Cin > 0 && Cout > 0 && k > 0 && stride > 0,
                "act_conv_transpose1d_fused: bad argument");
    ST2_REQUIRE(precision == ST2_PREC_BF16 || precision == ST2_PREC_FP16, "act_conv_transpose1d_fused: 16-bit precisions only");
    ST2_REQUIRE(k % stride == 0, "act_conv_transpose1d_fused: k must be a multiple of stride");
    ST2_REQUIRE((h_next == nullptr) == (coef_next == nullptr), "act_conv_transpose1d_fused: h_next and coef_next go together");
    cudaStream_t st = (cudaStream_t)stream;
    int64_t off[5];
    fused_t_offsets(B, Tin, Cin, Cout, k, stride, off);
    char* base = (char*)scratch;
    float* wp = (float*)(base + off[0]);
    void* w16 = base + off[1];
    float* coef = (float*)(base + off[2]);
    void* parts = base + off[3];
    const int dt = precision == ST2_PREC_BF16 ? DT_BF16 : DT_F16;
    const int cin_pad = (Cin + 63) / 64 * 64, cout_pad = (Cout + 31) / 32 * 32;
    int e = launch_fold_pack(nullptr, w, wp, Cin, Cout, k, 1, st);
    if (e != ST2_OK) return e;
    e = launch_pack_w16(wp, w16, k, Cin, Cout, cin_pad, cout_pad, dt, st);
    if (e != ST2_OK) return e;
    e = launch_adain_coef(nullptr, nullptr, 0, 0, coef, B, Tin, Cin, Cin, st);
    if (e != ST2_OK) return e;
    ConvArgs a;
    memset(&a, 0, sizeof(a));
    a.B = B; a.Cin = Cin; a.Cout = Cout; a.Tin = Tin;
    a.Tout = (Tin - 1) * stride - 2 * padding + (k - 1) + output_padding + 1;
    ST2_REQUIRE(a.Tout > 0, "act_conv_transpose1d_fused: empty output");
    a.x = x; a.ld_x = Cin; a.w = wp; a.w16 = w16; a.w16_cin_pad = cin_pad; a.w16_cout_pad = cout_pad; a.fmt16 = dt;
    a.bias = bias; a.res = res; a.ld_res = Cout; a.y = y; a.ld_y = Cout;
    a.ntaps = k / stride; a.tap_step = -1; a.in_off = 0; a.in_stride = 1;
    a.phases = stride; a.w_step = stride; a.out_stride = stride; a.out_pad = padding;
    a.M = (a.Tout - 1 + padding) / stride + 1;
    a.scale = 1.f;
    ST2_REQUIRE(conv_fused_supported(a), "act_conv_transpose1d_fused: geometry not supported by the fused kernels");
    e = launch_conv_fused(a, coef, Cin, act, slope, alpha, h_next ? parts : nullptr, st);
    if (e != ST2_OK) return e;
    if (h_next != nullptr) e = launch_adain_coef_f2(parts, fused_stats_parts(a), h_next, 2 * Cout, 0, coef_next, B, a.Tout, Cout, Cout, st);
    return e;
}

// st2_act_conv_transpose1d_fused with the fp16 output of the decoder's upsampling step (decoder.cu, fp16_xu): with y16 the
// stage input is written as fp16 and widened into y.
int64_t st2_act_conv_transpose1d_fused_ex_scratch_bytes(int32_t B, int32_t Tin, int32_t Cin, int32_t Cout, int32_t k,
                                                        int32_t stride) {
    if (B <= 0 || Tin <= 0 || Cin <= 0 || Cout <= 0 || k <= 0 || stride <= 0) return ST2_ERR_INVALID;
    int64_t off[5];
    const int64_t Tmax = (int64_t)Tin * stride + k;               // >= Tout for any padding >= 0, output_padding < stride
    return fused_t_offsets(B, Tin, Cin, Cout, k, stride, off) + align256((int64_t)B * Tmax * Cout * 2);   // + y as fp16
}

int st2_act_conv_transpose1d_fused_ex(const float* x, const float* alpha, int32_t act, float slope, const float* w,
                                      const float* bias, const float* res, float* y, const float* h_next, float* coef_next,
                                      void* scratch, int32_t B, int32_t Tin, int32_t Cin, int32_t Cout, int32_t k,
                                      int32_t stride, int32_t padding, int32_t output_padding, int32_t y16, int32_t precision,
                                      void* stream) {
    ST2_REQUIRE(x && w && y && scratch && B > 0 && Tin > 0 && Cin > 0 && Cout > 0 && k > 0 && stride > 0 && padding >= 0 &&
                    output_padding >= 0 && output_padding < stride,
                "act_conv_transpose1d_fused_ex: bad argument");
    ST2_REQUIRE(precision == ST2_PREC_BF16 || precision == ST2_PREC_FP16, "act_conv_transpose1d_fused_ex: 16-bit precisions only");
    ST2_REQUIRE(k % stride == 0, "act_conv_transpose1d_fused_ex: k must be a multiple of stride");
    ST2_REQUIRE((h_next == nullptr) == (coef_next == nullptr), "act_conv_transpose1d_fused_ex: h_next and coef_next go together");
    cudaStream_t st = (cudaStream_t)stream;
    int64_t off[5];
    fused_t_offsets(B, Tin, Cin, Cout, k, stride, off);
    char* base = (char*)scratch;
    float* wp = (float*)(base + off[0]);
    void* w16 = base + off[1];
    float* coef = (float*)(base + off[2]);
    void* parts = base + off[3];
    void* y16b = base + off[4];
    const int dt = precision == ST2_PREC_BF16 ? DT_BF16 : DT_F16;
    const int cin_pad = (Cin + 63) / 64 * 64, cout_pad = (Cout + 31) / 32 * 32;
    int e = launch_fold_pack(nullptr, w, wp, Cin, Cout, k, 1, st);
    if (e == ST2_OK) e = launch_pack_w16(wp, w16, k, Cin, Cout, cin_pad, cout_pad, dt, st);
    if (e == ST2_OK) e = launch_adain_coef(nullptr, nullptr, 0, 0, coef, B, Tin, Cin, Cin, st);
    if (e != ST2_OK) return e;
    ConvArgs a;
    memset(&a, 0, sizeof(a));
    a.B = B; a.Cin = Cin; a.Cout = Cout; a.Tin = Tin;
    a.Tout = (Tin - 1) * stride - 2 * padding + (k - 1) + output_padding + 1;
    ST2_REQUIRE(a.Tout > 0, "act_conv_transpose1d_fused_ex: empty output");
    a.x = x; a.ld_x = Cin; a.w = wp; a.w16 = w16; a.w16_cin_pad = cin_pad; a.w16_cout_pad = cout_pad; a.fmt16 = dt;
    a.bias = bias; a.res = res; a.ld_res = Cout; a.y = y16 ? (float*)y16b : y; a.ld_y = Cout; a.y16out = y16 ? 1 : 0;
    a.ntaps = k / stride; a.tap_step = -1; a.in_off = 0; a.in_stride = 1;
    a.phases = stride; a.w_step = stride; a.out_stride = stride; a.out_pad = padding;
    a.M = (a.Tout - 1 + padding) / stride + 1;
    a.scale = 1.f;
    ST2_REQUIRE(conv_fused_supported(a), "act_conv_transpose1d_fused_ex: geometry not supported by the fused kernels");
    ST2_REQUIRE(!y16 || conv_pipe_supported(a),
                "act_conv_transpose1d_fused_ex: an fp16 output needs the TMA pipeline kernel, which cannot run this geometry");
    e = launch_conv_fused(a, coef, Cin, act, slope, alpha, h_next ? parts : nullptr, st);
    if (e == ST2_OK && y16) e = launch_half_to_float(y16b, y, (int64_t)B * a.Tout * Cout, st);
    if (e == ST2_OK && h_next != nullptr)
        e = launch_adain_coef_f2(parts, fused_stats_parts(a), h_next, 2 * Cout, 0, coef_next, B, a.Tout, Cout, Cout, st);
    return e;
}

}  // extern "C"
