/*
 * st2_b200.h -- C ABI of the B200-native StyleTTS2-lite waveform Decoder hot path.
 *
 * The reference (thewh1teagle/StyleTTS2-lite) has no FFI / plugin API for this path:
 * the boundary is the nn.Module duck-type `Decoder.forward(asr, F0_curve, N, s)` picked
 * by name in models.py:538-561 / inference.py:95-118 and called at inference.py:270.
 * These entry points are what a ctypes binding for that call (and for the length
 * regulation of inference.py:257-268) binds; styletts2_lite_b200/decoder.py is that
 * binding, INTEGRATION.md shows the three lines a reference maintainer changes.
 *
 * Conventions
 *   - every function returns 0 on success or a negative st2_status; nothing throws,
 *     exits or prints.  st2_last_error() returns a thread-local message.
 *   - all pointers named dev_* / asr / f0 / ... are raw DEVICE pointers owned by the
 *     caller (PyTorch).  No hidden allocation and no synchronisation happens inside
 *     st2_decoder_forward: the launches are ordered on the caller's stream and scratch
 *     comes from the caller-provided workspace.  (st2_decoder_finalize allocates the
 *     re-packed weights once; st2_decoder_destroy frees them.)
 *   - `stream` is a cudaStream_t passed as void*.
 *   - internal activations are channels-last fp32 [B][T][C]; the ABI itself speaks the
 *     reference's layouts (asr [B,512,T], F0_curve [B,2T], N [B,2T], s [B,128],
 *     out [B,1,600T]).
 */
#ifndef ST2_B200_H
#define ST2_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ST2_ABI_VERSION 1

#if defined(__GNUC__)
#define ST2_API __attribute__((visibility("default")))
#else
#define ST2_API
#endif

typedef enum {
    ST2_OK = 0,
    ST2_ERR_INVALID = -1,      /* bad argument / unknown name / shape mismatch */
    ST2_ERR_STATE = -2,        /* call order (e.g. forward before finalize) */
    ST2_ERR_CUDA = -3,         /* a CUDA runtime / driver call failed */
    ST2_ERR_WORKSPACE = -4,    /* workspace too small */
    ST2_ERR_UNSUPPORTED = -5   /* shape family or device not supported */
} st2_status;

/* arithmetic of the dense convolutions */
typedef enum {
    ST2_PREC_FP32 = 0,         /* SIMT FFMA, fp32 everywhere (parity backbone, <=1e-4) */
    ST2_PREC_BF16 = 1,         /* tcgen05 kind::f16, bf16 operands, fp32 accumulate in TMEM */
    ST2_PREC_FP16 = 2          /* tcgen05 kind::f16, fp16 operands, fp32 accumulate in TMEM */
} st2_precision;

/* Mirrors the `decoder:` block of Configs/config_example.yaml:57-73 plus the two
 * constructor arguments Decoder actually uses (dim_in, style_dim; hifigan.py:417-422,
 * istftnet.py:661-667). */
typedef struct {
    int32_t variant;                 /* 0 = hifigan, 1 = istftnet, 4 = vocos (2 / 3 are the predictor / text-encoder handles) */
    int32_t dim_in;                  /* 512 */
    int32_t style_dim;               /* 128 */
    int32_t upsample_initial_channel;/* 512 */
    int32_t n_stages;                /* len(upsample_rates): 4 (hifigan) / 2 (istftnet) */
    int32_t upsample_rates[4];
    int32_t upsample_kernel_sizes[4];
    int32_t n_kernels;               /* len(resblock_kernel_sizes) = 3 */
    int32_t resblock_kernel_sizes[3];
    int32_t resblock_dilations[3][3];
    int32_t gen_istft_n_fft;         /* 20 (istftnet), 1200 (vocos) */
    int32_t gen_istft_hop_size;      /* 5  (istftnet), 300 (vocos) */
    int32_t intermediate_dim;        /* vocos only: 1536 (config_example.yaml:76) */
    int32_t num_layers;              /* vocos only: 8 ConvNeXt blocks (config_example.yaml:77) */
} st2_config;

typedef struct st2_decoder st2_decoder;

ST2_API int st2_abi_version(void);
ST2_API const char* st2_last_error(void);

/* ---- Decoder: replaces Modules/hifigan.py:416-475 and Modules/istftnet.py:660-721 ---- */

/* Decoder.__init__ */
ST2_API int st2_decoder_create(const st2_config* cfg, st2_decoder** out);
ST2_API void st2_decoder_destroy(st2_decoder* d);

/* load_state_dict (inference.py:160): hand over one tensor of the reference state_dict by
 * its reference key ("generator.ups.0.weight_v", "encode.norm1.fc.bias", ...).  fp32,
 * contiguous, on the device; only read during st2_decoder_finalize. */
ST2_API int st2_decoder_set_weight(st2_decoder* d, const char* name, const float* dev_ptr,
                           const int64_t* shape, int32_t ndim);

/* Fold weight-norm (w = v*g/||v||, norm over all dims but 0), transpose every conv to the
 * tap-major [k][Cin][Cout] layout, build bf16/fp16 copies for the tensor-core path and
 * concatenate the 106 (hifigan) AdaIN fc layers into one [R,128] matrix.  Allocates the
 * packed weights (device) and synchronises `stream` once. */
ST2_API int st2_decoder_finalize(st2_decoder* d, void* stream);

/* number of parameters handed over (the reference prints it, inference.py:170-171) */
ST2_API int64_t st2_decoder_num_params(const st2_decoder* d);

/* scratch needed by one forward of B utterances x T asr frames at `precision` */
ST2_API int64_t st2_decoder_workspace_bytes(const st2_decoder* d, int32_t B, int32_t T, int32_t precision);

/* Decoder.forward(asr, F0_curve, N, s) in eval mode.
 *   asr [B,dim_in,T]  f0 [B,2T]  n [B,2T]  s [B,style_dim]  ->  out [B,1,spf*T]
 *   (spf = 600 samples per asr frame for both shipped variants).
 *   noise: the SineGen `randn_like` draw (hifigan.py:213), [B,spf*T,9] fp32, or NULL to
 *   draw it on the device from Philox4x32-10 keyed by `seed` (the reference uses the
 *   global torch RNG; the two other draws, hifigan.py:126 and :267, never reach the
 *   output -- SURVEY.md 8(a)). */
ST2_API int st2_decoder_forward(st2_decoder* d, const float* asr, const float* f0, const float* n,
                        const float* s, const float* noise, uint64_t seed, float* out,
                        int32_t B, int32_t T, int32_t precision,
                        void* workspace, int64_t workspace_bytes, void* stream);

/* Debug / per-layer parity: copy the named intermediate of the NEXT forwards into dst as a
 * dense channels-last fp32 [B][T'][C] (capacity in floats; dst=NULL unregisters).  Names
 * follow the oracle's taps ("encode", "decode.3", "har_source",
 * "generator.resblocks.5.iter2", "generator.stage1.out", ...). */
ST2_API int st2_decoder_set_tap(st2_decoder* d, const char* name, float* dst, int64_t capacity);

/* Options of the 16-bit precisions.  "fp16_storage" (default 1): keep the stage-private tensors of the generator (conv1
 * output and running tensor of AdaINResBlock1, stage input, partial sum over the resblocks) in fp16 between kernels --
 * a third fewer HBM bytes for ~0.4 dB of SNR (DESIGN.md section 3); 0 stores every tensor as fp32.  "fp16_xt", "fp16_run",
 * "fp16_xu", "fp16_sum" (default 1 each) switch the four kinds of tensors individually.  Unknown names fail. */
ST2_API int st2_decoder_set_option(st2_decoder* d, const char* name, int32_t value);

/* Process-wide test hooks: "no_pipe", "row_always", "row_sub", "no_row_inline_coef", "verbose" (default 0 each); unknown names
 * fail.  Not synchronised: call it while no forward is running. */
ST2_API int st2_set_tuning(const char* name, int32_t value);

/* Optional device-resident Philox seed: when set (non-NULL), the harmonic source reads its noise seed from *dev_seed
 * at run time instead of the `seed` argument of st2_decoder_forward, so a forward captured in a CUDA graph
 * (the forward allocates nothing and never synchronises) draws new noise on every replay.  NULL restores `seed`. */
ST2_API int st2_decoder_set_seed_buffer(st2_decoder* d, const uint64_t* dev_seed);

/* how many kernels of this library the last forward launched */
ST2_API int64_t st2_decoder_last_launch_count(const st2_decoder* d);

/* Per-launch event profile (bench.py's roofline leg).  With profiling enabled every forward
 * records one CUDA event after each kernel launch on the caller's stream; get_profile waits
 * for the last one and returns, per kernel category, the summed device time (ms), the launch
 * count and the ALGORITHMIC flops / bytes (SURVEY.md 8(d) figures) of those launches.
 * Arrays must hold st2_profile_num_categories() entries. */
ST2_API int st2_decoder_set_profiling(st2_decoder* d, int32_t enable);
ST2_API int st2_profile_num_categories(void);
ST2_API const char* st2_profile_category_name(int32_t cat);
ST2_API int st2_decoder_get_profile(st2_decoder* d, double* ms, int64_t* launches, double* flops,
                            double* bytes);

/* the same profile per launch, in launch order; returns the number of records written */
ST2_API int64_t st2_decoder_get_profile_launches(st2_decoder* d, int64_t max_n, int32_t* cat, float* ms,
                                         double* flops, double* bytes);

/* ---- F0 / energy predictor (SURVEY.md 8(f) N1): replaces ProsodyPredictor.F0Ntrain, models.py:448-461 ----
 * The step right before the Decoder (inference.py:267): shared bidirectional LSTM (models.py:407), two stacks of
 * three AdainResBlk1d (models.py:408-416) and two 1x1 projections (models.py:418-419).  The handle is an st2_decoder
 * of a third kind: st2_decoder_set_weight (keys "shared.weight_ih_l0", "F0.1.conv1.weight_v", "N_proj.bias", ...
 * as in ProsodyPredictor.state_dict()), st2_decoder_finalize, st2_decoder_set_tap, the profile calls and
 * st2_decoder_destroy apply unchanged; st2_decoder_forward / _workspace_bytes reject it. */
ST2_API int st2_f0n_create(int32_t d_hid, int32_t style_dim, st2_decoder** out);
ST2_API int64_t st2_f0n_workspace_bytes(const st2_decoder* d, int32_t B, int32_t T, int32_t precision);
/* en [B, d_hid+style_dim, T] (the length-regulated DurationEncoder output), s [B, style_dim]
 *   -> f0 [B, 2T], n [B, 2T]   (what Decoder.forward takes as F0_curve and N).
 * precision: fp32 = SIMT everywhere; bf16 / fp16 = the convolutions and the LSTM input projection on tcgen05 with
 * fp16 operands (the recurrence itself is always fp32). */
ST2_API int st2_f0n_forward(st2_decoder* d, const float* en, const float* s, float* f0, float* n, int32_t B, int32_t T,
                    int32_t precision, void* workspace, int64_t workspace_bytes, void* stream);

/* Duration half of the same predictor (SURVEY.md 8(f) N2): replaces inference.py:242-245 --
 *   d = predictor.text_encoder(t_en, s, lengths, mask)        DurationEncoder.forward, models.py:485-520
 *   x, _ = predictor.lstm(d) ; duration = sigmoid(predictor.duration_proj(x)).sum(-1)
 * for a batch of equal-length utterances (st2_dur_forward_ragged below takes padded ones).  Available when the handle was also
 * given the reference keys
 * "text_encoder.lstms.*", "lstm.*" and "duration_proj.linear_layer.*" before st2_decoder_finalize.
 *   t_en [B, d_hid, L], s [B, style_dim]  ->  d [B, L, d_hid+style_dim] (the reference's layout), duration [B, L]
 * (feed `duration` to st2_round_durations and `d`, transposed, to st2_length_regulate). */
ST2_API int64_t st2_dur_workspace_bytes(const st2_decoder* d, int32_t B, int32_t L, int32_t precision);
ST2_API int st2_dur_forward(st2_decoder* d, const float* t_en, const float* s, float* d_out, float* duration, int32_t B,
                    int32_t L, int32_t precision, void* workspace, int64_t workspace_bytes, void* stream);
/* The same call for a PADDED batch, as ProsodyPredictor.forward runs it (models.py:422-442): lengths [B] int32 on the device,
 * 0 <= lengths[b] <= L (nullptr = st2_dur_forward).  Rows of `d` behind an utterance are zero (the masked_fill_ calls of
 * models.py:491, :500), every LSTM is the pack_padded_sequence one (models.py:503-509, :426-435: the reverse direction of
 * utterance b starts at token lengths[b]-1), and `duration` at a padded token is what duration_proj makes of a zero row, as in
 * the reference.  Utterance b of the result equals the B = 1 call on its first lengths[b] tokens. */
ST2_API int st2_dur_forward_ragged(st2_decoder* d, const float* t_en, const float* s, const int32_t* lengths, float* d_out,
                    float* duration, int32_t B, int32_t L, int32_t precision, void* workspace, int64_t workspace_bytes,
                    void* stream);

/* ---- TextEncoder (SURVEY.md 8(f) N3): replaces models.py:238-285, called at inference.py:239 ----
 * nn.Embedding -> depth x [weight-normed Conv1d(k) -> LayerNorm over channels -> LeakyReLU(0.2)] -> bidirectional LSTM, for a
 * batch of equal-length token sequences.  Same handle type and weight / finalize / tap / destroy calls as above; keys as in
 * TextEncoder.state_dict() ("embedding.weight", "cnn.0.0.weight_v", "cnn.0.1.gamma", "lstm.weight_hh_l0_reverse", ...).
 *   tokens [B, L] int64 (device)  ->  out [B, channels, L]  (= t_en, the input of st2_dur_forward and st2_length_regulate) */
ST2_API int st2_text_create(int32_t channels, int32_t kernel_size, int32_t depth, int32_t n_symbols, st2_decoder** out);
ST2_API int64_t st2_text_workspace_bytes(const st2_decoder* d, int32_t B, int32_t L, int32_t precision);
ST2_API int st2_text_forward(st2_decoder* d, const int64_t* tokens, float* out, int32_t B, int32_t L, int32_t precision,
                     void* workspace, int64_t workspace_bytes, void* stream);
/* The same call for a PADDED batch (TextEncoder.forward with a non-trivial mask m, models.py:258-285): lengths [B] int32 on the
 * device, 0 <= lengths[b] <= L (nullptr = st2_text_forward).  Tokens behind an utterance are zeroed after the embedding and after
 * every cnn block (models.py:262, :266), the LSTM is the packed one (models.py:270-277), columns l >= lengths[b] of `out` are
 * zero (models.py:279-283). */
ST2_API int st2_text_forward_ragged(st2_decoder* d, const int64_t* tokens, const int32_t* lengths, float* out, int32_t B, int32_t L,
                    int32_t precision, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- Duration smoothing: replaces inference.py:248-255 (+ the mean returned at :272) ----
 * Per utterance b, over its n_tokens[b] tokens (nullptr = L):
 *   mu  = prev_d_mean[b] if it is non-zero else mean(duration_b);  sd = std(duration_b)          (unbiased, inference.py:248-251)
 *   dur = duration * (1 - t) + (noise * sd + mu) * t                                             (inference.py:252)
 *   dur[1:-2] <- mean + sign * 3 * 0.95 * std of that slice wherever |z-score| > 3               (inference.py:253, :134-148)
 *   dur /= speed ;  mean_out[b] = mean(dur)                                                      (inference.py:255, :272)
 * noise [B, L] is the caller's N(0, 1) tape standing in for torch.Tensor.normal_ (null allowed when t == 0); prev_d_mean [B] and
 * mean_out [B] may be null.  Tokens beyond n_tokens[b] are written as 0.  All pointers are device memory; feed `out` to
 * st2_round_durations. */
ST2_API int st2_smooth_durations(const float* duration, const int32_t* n_tokens, const float* noise, const float* prev_d_mean,
                        float t, float speed, float* out, float* mean_out, int32_t B, int32_t L, void* stream);
/* The same for the B sentences of one text in order, as the loop of StyleTTS2.generate chains them (inference.py:312-313): sentence
 * b takes the mean duration of sentence b - 1 (mean_out[b - 1]) as its prev_d_mean; prev_d_mean0 (device, 1 float, may be null = 0)
 * seeds sentence 0. */
ST2_API int st2_smooth_durations_chained(const float* duration, const int32_t* n_tokens, const float* noise,
                        const float* prev_d_mean0, float t, float speed, float* out, float* mean_out, int32_t B, int32_t L,
                        void* stream);

/* ---- Length regulator: replaces inference.py:257-268 ---- */

/* torch.round (half to even) + clamp(min=1) of the predicted durations (inference.py:257);
 * tokens at or beyond n_tokens[b] get 0.  duration [B,L] fp32 -> dur [B,L] int32,
 * total_frames [B] int32. */
ST2_API int st2_round_durations(const float* duration, const int32_t* n_tokens, int32_t* dur,
                        int32_t* total_frames, int32_t B, int32_t L, void* stream);

/* out[b,c,f] = src[b,c,tok_b(f)] for f < sum(dur[b,:]), 0 beyond: the `src @ alignment`
 * products of inference.py:266 and :268 as a bit-exact gather (the one-hot matmul adds
 * only zeros).  src [B,C,L], dur [B,L] int32 (>=0), out [B,C,F].  channels_last != 0
 * writes out as [B,F,C] instead (the decoder's internal layout). */
ST2_API int st2_length_regulate(const float* src, const int32_t* dur, float* out, int32_t B, int32_t C,
                        int32_t L, int32_t F, int32_t channels_last, void* stream);

/* ---- unit entry points (per-kernel parity, SURVEY.md 8(b)) ---- */

/* SineGen phase argument (hifigan.py:117-157): f0 [B,L2] -> phase [B,L2*scale,9],
 * bit-exact with the CPU reference.  frames_scratch: [B,L2,9] fp32. */
ST2_API int st2_sinegen_phase(const float* f0, float* phase, float* frames_scratch, int32_t B, int32_t L2,
                      int32_t upsample_scale, void* stream);

/* SourceModuleHnNSF.forward (hifigan.py:254-268): f0 [B,L2] -> har_source [B,L2*scale].
 * lin_w [9], lin_b [1] device pointers; noise as in st2_decoder_forward. */
ST2_API int st2_har_source(const float* f0, const float* noise, uint64_t seed, const float* lin_w,
                   const float* lin_b, float* har, float* frames_scratch, int32_t B, int32_t L2,
                   int32_t upsample_scale, void* stream);

/* generator.noise_convs[i] (hifigan.py:296-303,330) on the harmonic source, as the decoder runs it: har [B,S] ->
 * y [B,Tout,C] channels-last, Tout = (S + 2*pad - k)/stride + 1, w [C,1,k] (reference layout), bias [C].  y is fp32, or with
 * y16 fp16 WITHOUT the bias (the decoder's fp16 noise source).  If h [B,2C] is given, coef [B,2,C] receives the AdaIN
 * coefficients (a = (1+gamma)*rstd, b = beta - mean*a) of the conv output from the kernel's statistics partials, with b
 * for the tensor as stored (mean taken without the bias when y16).  scratch: st2_noise_conv_scratch_bytes(...) bytes. */
ST2_API int64_t st2_noise_conv_scratch_bytes(int32_t B, int32_t Tout, int32_t C, int32_t k, int32_t stride);
ST2_API int st2_noise_conv(const float* har, const float* w, const float* bias, void* y, const float* h, float* coef,
                   void* scratch, int32_t B, int32_t S, int32_t Tout, int32_t C, int32_t k, int32_t stride, int32_t pad,
                   int32_t y16, void* stream);

/* Generator tail (hifigan.py:343-345): out [B,S] = tanh(conv_post(snake(x, alpha))), conv_post C -> 1, k = 7, padding 3.
 * x [B,S,C] channels-last with row pitch ld_x (a multiple of 4), fp32, or fp16 when x16 (needs fast); C a multiple of 4,
 * <= 64.  w [1,C,7] (reference layout), bias [1], alpha [C].  fast selects __sinf / __fdividef (the 16-bit precisions).
 * w_scratch: 7*C floats receiving the packed weight. */
ST2_API int st2_post_hifigan(const void* x, int32_t ld_x, const float* alpha, const float* w, const float* bias, float* out,
                     float* w_scratch, int32_t B, int32_t S, int32_t C, int32_t fast, int32_t x16, void* stream);

/* All AdaIN fc layers of a decoder in one launch (hifigan.py:18,21): h [B,R] = s [B,K] @ W[R,K]^T + bias [R].
 * K a multiple of 4, <= 1024. */
ST2_API int st2_style_fc(const float* s, const float* W, const float* bias, float* h, int32_t B, int32_t R, int32_t K,
                 void* stream);

/* AdaIN1d + activation (hifigan.py:14-24 with :68 or LeakyReLU) on channels-last
 * x [B,T,C] (pitch ld_x): y = act((1+gamma)*IN(x)+beta), gamma|beta = h[b, 0:C | C:2C].
 * act: 0 none, 1 leaky-relu(slope), 2 snake(alpha[C]).  out_dtype: 0 fp32, 1 bf16, 2 fp16.
 * scratch: at least st2_adain_scratch_bytes(B,T,C) bytes. */
ST2_API int64_t st2_adain_scratch_bytes(int32_t B, int32_t T, int32_t C);
ST2_API int st2_adain_act(const float* x, int32_t ld_x, const float* h, int32_t ld_h, const float* alpha,
                  int32_t act, float slope, void* y, int32_t ld_y, int32_t out_dtype,
                  int32_t B, int32_t T, int32_t C, void* scratch, void* stream);

/* Conv1d / ConvTranspose1d on channels-last fp32 x [B,Tin,Cin] with the reference weight
 * layout (Conv1d [Cout,Cin,k]; ConvTranspose1d [Cin,Cout,k]); y [B,Tout,Cout].
 * transposed != 0 selects ConvTranspose1d (stride = upsampling factor).  scratch holds the
 * re-packed weight (and, for 16-bit precisions, the 16-bit operand copies):
 * st2_conv1d_scratch_bytes(...) bytes. */
ST2_API int64_t st2_conv1d_scratch_bytes(int32_t B, int32_t Tin, int32_t Cin, int32_t Cout, int32_t k,
                                 int32_t precision);
ST2_API int st2_conv1d(const float* x, const float* w, const float* bias, float* y, void* scratch,
               int32_t B, int32_t Tin, int32_t Cin, int32_t Cout, int32_t k, int32_t stride,
               int32_t padding, int32_t dilation, int32_t output_padding, int32_t transposed,
               int32_t precision, void* stream);

/* SURVEY.md 8(f) N4 -- waveform post-processing and wire format, the step after the path:
 *   StyleTTS2.generate, inference.py:314-319:  wav_i = wav_i[trim:-trim] (trim = 4000) for every sentence, concatenate,
 *                                              pad `pad` (= 4000) zeros on both sides (float64 from here on);
 *   Demo/infer.py:51-54:                       r = r / max|r|;  soundfile.write(..., 24000) -> PCM_16 = lrint(r * 32767)
 *                                              (libsndfile pcm.c d2s_array; soundfile 0.13.1, uv.lock:1925).
 * wav [B,S] fp32 device tensor (the decoder output of one batch of sentences), lengths [B] int32 device (samples of each
 * sentence, NULL: all S).  out_f64 / out_pcm (either may be NULL) need st2_postprocess_max_samples() elements; *out_total
 * (device int64) receives the number of samples written.  Bit-exact against the numpy restatement (oracle/postprocess_np.py).
 * An all-zero input gives zeros (the reference would divide by zero). */
ST2_API int64_t st2_postprocess_scratch_bytes(int32_t B);
ST2_API int64_t st2_postprocess_max_samples(int32_t B, int32_t S, int32_t trim, int32_t pad);
ST2_API int st2_postprocess(const float* wav, const int32_t* lengths, int32_t B, int32_t S, int32_t trim, int32_t pad,
                    double* out_f64, int16_t* out_pcm, int64_t* out_total, void* scratch, void* stream);

/* One fused half-step of AdaINResBlock1 (Modules/hifigan.py:67-73) on channels-last fp32 tensors, through the
 * tensor-core fused kernels (16-bit operands, fp32 accumulate):
 *   y = (conv1d(act(AdaIN(x; h)), w) + bias + res (+ y_old if accumulate)) * scale
 * h [B,2*Cin] (NULL: no normalisation), alpha [Cin] for snake, w [Cout,Cin,k] (2*padding == dilation*(k-1)),
 * res [B,T,Cout] or NULL.  If h_next [B,2*Cout] is given, coef_next [B,2,Cout] receives the AdaIN coefficients
 * (a = (1+gamma)*rstd, b = beta - mean*a) of y computed from the epilogue's statistics partials. */
ST2_API int64_t st2_adain_conv1d_fused_scratch_bytes(int32_t B, int32_t T, int32_t Cin, int32_t Cout, int32_t k);
ST2_API int st2_adain_conv1d_fused(const float* x, const float* h, const float* alpha, int32_t act, float slope,
                           const float* w, const float* bias, const float* res, float* y, const float* h_next,
                           float* coef_next, void* scratch, int32_t B, int32_t T, int32_t Cin, int32_t Cout,
                           int32_t k, int32_t padding, int32_t dilation, float scale, int32_t accumulate,
                           int32_t precision, void* stream);

/* st2_adain_conv1d_fused with the fp16 storage types of the decoder's resblocks (Modules/hifigan.py:65-74, :338-342): x is
 * stored as fp16 when x16, res when res16, y is written as fp16 and widened when y16.  old [B,T,Cout] (may be NULL, needs
 * accumulate) is a separate accumulate source replacing the old values in y, stored as fp16 when old16; with old_in_y (needs
 * old16 and y16) it is first stored into the fp16 y buffer and the conv accumulates in place, as the middle resblock of a
 * stage updates the fp16 stage sum.  All pointers are fp32 channels-last tensors; the conversions happen in scratch.
 *   y = (conv1d(act(AdaIN(x; h)), w) + bias + res + old) * scale
 * Any 16-bit flag needs a geometry the TMA pipeline kernel runs; otherwise ST2_ERR_INVALID. */
ST2_API int64_t st2_adain_conv1d_fused_ex_scratch_bytes(int32_t B, int32_t T, int32_t Cin, int32_t Cout, int32_t k);
ST2_API int st2_adain_conv1d_fused_ex(const float* x, const float* h, const float* alpha, int32_t act, float slope,
                              const float* w, const float* bias, const float* res, const float* old, float* y,
                              const float* h_next, float* coef_next, void* scratch, int32_t B, int32_t T, int32_t Cin,
                              int32_t Cout, int32_t k, int32_t padding, int32_t dilation, float scale, int32_t accumulate,
                              int32_t x16, int32_t res16, int32_t old16, int32_t y16, int32_t old_in_y, int32_t precision,
                              void* stream);

/* The same half-step (Snake, C = Cin = Cout in {32, 64}) on the row-per-thread kernel with the storage types of the 16-bit
 * decoder paths: res / old (the running tensor and the partial stage sum of Modules/hifigan.py:65-74, :338-342) are stored as
 * fp16 and added by the tensor core; x is stored as fp16 when x16, y is written as fp16 when y16.  All pointers are fp32
 * channels-last tensors; the conversions happen in scratch.  y = (conv1d(snake(AdaIN(x; h))) + bias + res + old) * scale. */
ST2_API int64_t st2_adain_conv1d_row_scratch_bytes(int32_t B, int32_t T, int32_t C, int32_t k);
ST2_API int st2_adain_conv1d_row(const float* x, const float* h, const float* alpha, const float* w, const float* bias,
                         const float* res, const float* old, float* y, const float* h_next, float* coef_next,
                         void* scratch, int32_t B, int32_t T, int32_t C, int32_t k, int32_t padding, int32_t dilation,
                         float scale, int32_t precision, int32_t x16, int32_t y16, void* stream);

/* Two chained half-steps on the row-per-thread kernel, as one iteration of AdaINResBlock1 (Modules/hifigan.py:67-73) runs them
 * in the decoder (x stored as fp16, padding dil * (k - 1) / 2):
 *   y1 = conv1d(snake(AdaIN(x; h1), alpha1), w1) + bias1                    (stored as fp16)
 *   y2 = conv1d(snake(AdaIN(y1; h2), alpha2), w2) + bias2 + x                (stored as fp16)
 * The second launch computes the AdaIN coefficients of y1 itself from the statistics partials of the first when its table of
 * them fits (<= 2 KB per CTA, and switch "no_row_inline_coef" off); otherwise the coefficient kernel runs between the two.
 * *inline_coef (host, may be NULL) receives 1 if the second launch computed them itself.  y1 / y2 [B,T,C] fp32 receive the
 * stored fp16 values widened; if h_next is given, coef_next [B,2,C] the AdaIN coefficients of y2. */
ST2_API int64_t st2_adain_conv1d_row_pair_scratch_bytes(int32_t B, int32_t T, int32_t C, int32_t k1, int32_t k2);
ST2_API int st2_adain_conv1d_row_pair(const float* x, const float* h1, const float* alpha1, const float* w1, const float* bias1,
                              const float* h2, const float* alpha2, const float* w2, const float* bias2, float* y1, float* y2,
                              const float* h_next, float* coef_next, int32_t* inline_coef, void* scratch, int32_t B, int32_t T,
                              int32_t C, int32_t k1, int32_t dil1, int32_t k2, int32_t dil2, int32_t precision, void* stream);

/* Generator upsampling step (Modules/hifigan.py:329-334) through the fused tensor-core kernels:
 *   y = conv_transpose1d(act(x), w) + bias + res        x [B,Tin,Cin], w [Cin,Cout,k] (k a multiple of stride),
 * res / y [B,Tout,Cout], Tout = (Tin-1)*stride - 2*padding + k + output_padding.  alpha [Cin] for snake.
 * If h_next [B,2*Cout] is given, coef_next [B,2,Cout] receives the AdaIN coefficients of y. */
ST2_API int64_t st2_act_conv_transpose1d_fused_scratch_bytes(int32_t B, int32_t Tin, int32_t Cin, int32_t Cout, int32_t k,
                                                     int32_t stride);
ST2_API int st2_act_conv_transpose1d_fused(const float* x, const float* alpha, int32_t act, float slope, const float* w,
                                   const float* bias, const float* res, float* y, const float* h_next,
                                   float* coef_next, void* scratch, int32_t B, int32_t Tin, int32_t Cin, int32_t Cout,
                                   int32_t k, int32_t stride, int32_t padding, int32_t output_padding,
                                   int32_t precision, void* stream);

/* st2_act_conv_transpose1d_fused with the fp16 output of the decoder's upsampling step: with y16, y is written as fp16 (the
 * stage input the resblocks read) and widened into the fp32 y; that needs a geometry the TMA pipeline kernel runs, otherwise
 * ST2_ERR_INVALID.  output_padding < stride. */
ST2_API int64_t st2_act_conv_transpose1d_fused_ex_scratch_bytes(int32_t B, int32_t Tin, int32_t Cin, int32_t Cout, int32_t k,
                                                        int32_t stride);
ST2_API int st2_act_conv_transpose1d_fused_ex(const float* x, const float* alpha, int32_t act, float slope, const float* w,
                                      const float* bias, const float* res, float* y, const float* h_next,
                                      float* coef_next, void* scratch, int32_t B, int32_t Tin, int32_t Cin, int32_t Cout,
                                      int32_t k, int32_t stride, int32_t padding, int32_t output_padding, int32_t y16,
                                      int32_t precision, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ST2_B200_H */
