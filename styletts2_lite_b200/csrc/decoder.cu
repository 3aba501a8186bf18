// Decoder handle, load-time weight packing and the forward "program" (the sequence of kernel
// launches that replaces Decoder.forward / Generator.forward, Modules/hifigan.py:446-475,
// :321-347 and Modules/istftnet.py:692-721, :542-573), plus the C ABI of include/st2_b200.h.
#include <stdarg.h>

#include "program.cuh"

namespace st2 {

thread_local char g_err[1024] = "";
thread_local int64_t g_launch_count = 0;

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

// Vocos generator weights (vocos.py:103-162: ConvNeXt blocks, final LayerNorm; :249-260: ISTFTHead.out and the ISTFT window)
static void pack_vocos_generator(st2_decoder* d, Packer& P) {
    const st2_config& c = d->cfg;
    const int dim = c.dim_in, inter = c.intermediate_dim, N = c.gen_istft_n_fft;
    for (int i = 0; i < c.num_layers; ++i) {
        const std::string n = "generator.convnext." + std::to_string(i);
        st2_decoder::ConvNeXtW& L = d->vx[i];
        ConvW dw;                                                    // depthwise Conv1d weight [dim,1,7] -> [7][dim]
        P.conv(dw, n + ".dwconv", 1, dim, 7, false, true, false);
        L.dw_w = dw.w32; L.dw_b = dw.bias;
        P.adain(L.norm, n + ".norm", dim);
        P.linear(L.pw1, n + ".pwconv1.weight", n + ".pwconv1.bias", dim, inter);
        const RawTensor* g = P.get(n + ".gamma");
        if (!g || g->numel() != dim) {
            if (P.err == ST2_OK) { set_error("%s.gamma must have %d elements", n.c_str(), dim); P.err = ST2_ERR_INVALID; }
            return;
        }
        P.linear(L.pw2, n + ".pwconv2.weight", n + ".pwconv2.bias", inter, dim, g->ptr);     // gamma * (W x + b), vocos.py:63-64
    }
    d->vx_ln = (float*)P.dalloc((size_t)2 * dim * sizeof(float));
    const float* lw = P.copy("generator.final_layer_norm.weight", dim);
    const float* lb = P.copy("generator.final_layer_norm.bias", dim);
    if (!d->vx_ln || !lw || !lb) return;
    if (cudaMemcpyAsync(d->vx_ln, lw, (size_t)dim * sizeof(float), cudaMemcpyDeviceToDevice, P.st) != cudaSuccess ||
        cudaMemcpyAsync(d->vx_ln + dim, lb, (size_t)dim * sizeof(float), cudaMemcpyDeviceToDevice, P.st) != cudaSuccess)
        P.err = ST2_ERR_CUDA;
    d->vx_kpad = round_up(N + 2, 128);                                // 1202 -> 1280: whole 256-column MMA tiles
    P.linear(d->vx_out, "generator.stft.out.weight", "generator.stft.out.bias", dim, N + 2, nullptr, d->vx_kpad);
    d->vx_window = P.copy("generator.stft.istft.window", N);
    ConvW& bs = d->vx_basis;
    bs.Cin = d->vx_kpad; bs.Cout = N; bs.k = 1; bs.transposed = false;
    bs.w32 = (float*)P.dalloc((size_t)d->vx_kpad * N * sizeof(float));
    if (!bs.w32 || !d->vx_window || P.err != ST2_OK) return;
    if (launch_vocos_basis(d->vx_window, bs.w32, N, d->vx_kpad, P.st) != ST2_OK) P.err = ST2_ERR_CUDA;
    if (d->tc_ok && N % 16 == 0) {
        bs.cin_pad = d->vx_kpad; bs.cout_pad = N;
        for (int dt = DT_BF16; dt <= DT_F16; ++dt) {
            bs.w16[dt] = P.dalloc((size_t)d->vx_kpad * N * 2);
            if (bs.w16[dt] && launch_pack_w16(bs.w32, bs.w16[dt], 1, d->vx_kpad, N, d->vx_kpad, N, dt, P.st) != ST2_OK) P.err = ST2_ERR_CUDA;
        }
    }
}

// Decoder weights (hifigan.py:416-443, istftnet.py:660-690; vocos.py:364-393)
static void pack_decoder(st2_decoder* d, Packer& P) {
    const st2_config& c = d->cfg;
    const int dim_in = c.dim_in;
    P.resblk1d(d->encode, "encode", dim_in + 2, 1024, false);
    for (int i = 0; i < 3; ++i) P.resblk1d(d->decode[i], "decode." + std::to_string(i), 1024 + 2 + 64, 1024, false);
    P.resblk1d(d->decode[3], "decode.3", 1024 + 2 + 64, c.upsample_initial_channel, true);
    {
        ConvW t;
        P.conv(t, "F0_conv", 1, 1, 3, false, true, false);
        d->f0_w = t.w32; d->f0_b = t.bias;
        ConvW u;
        P.conv(u, "N_conv", 1, 1, 3, false, true, false);
        d->n_w = u.w32; d->n_b = u.bias;
    }
    P.conv(d->asr_res, "asr_res.0", dim_in, 64, 1, false, true, true);
    if (c.variant == 4) {
        pack_vocos_generator(d, P);
        return;
    }
    d->lin_w = P.copy("generator.m_source.l_linear.weight", 9);
    d->lin_b = P.copy("generator.m_source.l_linear.bias", 1);
    const bool istft = c.variant == 1;
    const int c0 = c.upsample_initial_channel;
    if (!istft) d->gen_alpha[0] = P.copy("generator.alphas.0", c0);
    const int dil135[3] = {1, 3, 5};
    for (int i = 0; i < c.n_stages; ++i) {
        const int C = d->stage_channels(i);
        const std::string is = std::to_string(i);
        int sf = 1;
        for (int j = i + 1; j < c.n_stages; ++j) sf *= c.upsample_rates[j];
        const bool last = (i + 1 == c.n_stages);
        const int nc_cin = istft ? c.gen_istft_n_fft + 2 : 1;
        P.conv(d->noise_convs[i], "generator.noise_convs." + is, nc_cin, C, last ? 1 : 2 * sf, false, true, false);
        P.resblock1(d->noise_res[i], "generator.noise_res." + is, C, last ? 11 : 7, dil135);
        d->noise_c2b[i] = (float*)P.dalloc((size_t)C * sizeof(float));
        if (d->noise_c2b[i] && d->noise_res[i].c2[0].bias && d->noise_convs[i].bias && P.err == ST2_OK &&
            launch_add_vec(d->noise_c2b[i], d->noise_res[i].c2[0].bias, d->noise_convs[i].bias, C, P.st) != ST2_OK)
            P.err = ST2_ERR_CUDA;
        P.conv(d->ups[i], "generator.ups." + is, 2 * C, C, c.upsample_kernel_sizes[i], true, true, true);
        if (!istft) d->gen_alpha[i + 1] = P.copy("generator.alphas." + std::to_string(i + 1), C);
        for (int j = 0; j < c.n_kernels; ++j)
            P.resblock1(d->resblocks[i * c.n_kernels + j], "generator.resblocks." + std::to_string(i * c.n_kernels + j),
                        C, c.resblock_kernel_sizes[j], c.resblock_dilations[j]);
    }
    {
        const int Cl = d->stage_channels(c.n_stages - 1);
        P.conv(d->conv_post, "generator.conv_post", Cl, istft ? c.gen_istft_n_fft + 2 : 1, 7, false, true, istft);
    }
    if (istft) {
        const int n = c.gen_istft_n_fft, bins = n / 2 + 1;
        d->stft_fr = P.copy("generator.stft.weight_forward_real", (int64_t)bins * n);
        d->stft_fi = P.copy("generator.stft.weight_forward_imag", (int64_t)bins * n);
        d->stft_br = P.copy("generator.stft.weight_backward_real", (int64_t)bins * n);
        d->stft_bi = P.copy("generator.stft.weight_backward_imag", (int64_t)bins * n);
    }
}

static int finalize_impl(st2_decoder* d, cudaStream_t st) {
    const st2_config& c = d->cfg;
    Packer P{d, st};
    d->fc_rows = 0;
    if (c.variant == 2) pack_predictor(d, P);
    else if (c.variant == 3) pack_text_encoder(d, P);
    else pack_decoder(d, P);
    if (P.err != ST2_OK) return P.err;
    // all AdaIN fc layers -> one [R,style] matrix (rows: gamma(C) | beta(C) per instance)
    d->fc_w = (float*)P.dalloc((size_t)d->fc_rows * c.style_dim * sizeof(float));
    d->fc_b = (float*)P.dalloc((size_t)d->fc_rows * sizeof(float));
    if (!d->fc_w || !d->fc_b) return P.err;
    int row = 0;
    for (auto& pr : P.adain_list) {
        const RawTensor* w = P.get(pr.first + ".fc.weight");
        const RawTensor* b = P.get(pr.first + ".fc.bias");
        if (!w || !b) return P.err;
        const int rows = 2 * pr.second;
        if (w->numel() != (int64_t)rows * c.style_dim || b->numel() != rows) {
            set_error("AdaIN fc '%s' has the wrong shape", pr.first.c_str());
            return ST2_ERR_INVALID;
        }
        ST2_CUDA_CHECK(cudaMemcpyAsync(d->fc_w + (size_t)row * c.style_dim, w->ptr,
                                       (size_t)rows * c.style_dim * sizeof(float), cudaMemcpyDeviceToDevice, st));
        ST2_CUDA_CHECK(cudaMemcpyAsync(d->fc_b + row, b->ptr, (size_t)rows * sizeof(float), cudaMemcpyDeviceToDevice, st));
        row += rows;
    }
    ST2_CUDA_CHECK(cudaStreamSynchronize(st));
    ST2_CUDA_CHECK(cudaGetLastError());
    d->num_params = 0;
    for (auto& kv : d->raw)
        if (c.variant == 4 ? kv.first != "generator.stft.istft.window" : kv.first.find("generator.stft.") == std::string::npos)
            d->num_params += kv.second.numel();                       // registered buffers are not parameters
    d->finalized = true;
    return ST2_OK;
}

// Generator.forward + ISTFTHead.forward of the vocos variant (vocos.py:159-164, :268-296) on channels-last x [B][Tg][dim]
static void vocos_generator(Exec& E, st2_decoder* d, float* x, float* out, int Tg) {
    const st2_config& c = d->cfg;
    const int B = E.B, C = c.dim_in, I = c.intermediate_dim, N = c.gen_istft_n_fft, KP = d->vx_kpad;
    const int64_t rows = (int64_t)B * Tg;
    float* xa = x;
    float* xb = E.allocf(rows * C);
    float* yd = E.allocf(rows * C);
    float* hb = E.allocf(rows * I);
    void* a16 = E.alloc(rows * C * 4);
    void* g16 = E.alloc(rows * I * 4);
    for (int i = 0; i < c.num_layers; ++i) {
        const st2_decoder::ConvNeXtW& L = d->vx[i];
        const std::string name = "generator.convnext." + std::to_string(i);
        const int dt = E.fmt_for(name);
        if (E.live()) E.chk(launch_dwconv7(xa, L.dw_w, L.dw_b, yd, B, Tg, C, E.st));            // vocos.py:59
        E.prof(PC_MISC, 2.0 * rows * C * 7, 8.0 * rows * C);
        E.tap(name + ".dwconv", yd, C, rows, C);
        const bool tc1 = E.use_tc(L.pw1, dt), tc2 = E.use_tc(L.pw2, dt);
        E.norm_act(yd, C, Tg, C, &L.norm, ACT_NONE, 0.f, nullptr, a16, C, tc1 ? dt : DT_F32);   // vocos.py:60 (AdaIN1d)
        if (tc1 && tc2) {
            // 16-bit modes: GELU and the down-conversion in the first Linear's epilogue, no fp32 round trip of the 1536-wide tensor
            E.conv(L.pw1, a16, C, Tg, dt, (float*)g16, I, Tg, 1, 0, 1, nullptr, 0, 0, 1.f, 0, 0, 0, 1);   // vocos.py:62-63
        } else {
            E.conv(L.pw1, a16, C, Tg, tc1 ? dt : DT_F32, hb, I, Tg, 1, 0, 1, nullptr, 0, 0, 1.f, 0);   // vocos.py:62
            E.norm_act(hb, I, Tg, I, nullptr, ACT_GELU, 0.f, nullptr, g16, I, tc2 ? dt : DT_F32);   // vocos.py:63
        }
        E.conv(L.pw2, g16, I, Tg, tc2 ? dt : DT_F32, xb, C, Tg, 1, 0, 1, xa, C, 0, 1.f, 0);     // vocos.py:64-69 (gamma folded, + residual)
        std::swap(xa, xb);
        E.tap(name, xa, C, rows, C);
    }
    if (E.live()) E.chk(launch_layer_norm_lrelu(xa, d->vx_ln, d->vx_ln + C, 1.0f, yd, B, Tg, C, E.st, 1e-6f));   // vocos.py:162 (eps 1e-6)
    E.prof(PC_AFFINE_ACT, 0, 8.0 * rows * C);
    E.tap("generator.final_layer_norm", yd, C, rows, C);
    // ISTFTHead: the head GEMMs always take fp16 operands in the 16-bit modes (magnitudes up to 100 need the mantissa)
    const int dth = E.prec != ST2_PREC_FP32 ? DT_F16 : DT_F32;
    const bool tco = E.use_tc(d->vx_out, dth), tcb = E.use_tc(d->vx_basis, dth);
    E.norm_act(yd, C, Tg, C, nullptr, ACT_NONE, 0.f, nullptr, a16, C, tco ? dth : DT_F32);
    float* ob = E.allocf(rows * KP);
    E.conv(d->vx_out, a16, C, Tg, tco ? dth : DT_F32, ob, KP, Tg, 1, 0, 1, nullptr, 0, 0, 1.f, 0);   // vocos.py:280
    E.tap("generator.stft.out", ob, KP, rows, N + 2);
    void* sp = E.alloc(rows * KP * 4);
    if (E.live()) E.chk(launch_vocos_spec(ob, KP, sp, KP, tcb ? dth : DT_F32, rows, N / 2 + 1, E.st));   // vocos.py:281-292
    E.prof(PC_POST, 0, rows * KP * (4.0 + (tcb ? 2 : 4)));
    float* fr = E.allocf(rows * N);
    E.conv(d->vx_basis, sp, KP, Tg, tcb ? dth : DT_F32, fr, N, Tg, 1, 0, 1, nullptr, 0, 0, 1.f, 0);     // irfft * window, vocos.py:214-215
    if (E.live()) E.chk(launch_vocos_ola(fr, d->vx_window, out, B, Tg, N, c.gen_istft_hop_size, E.st));   // vocos.py:218-230
    E.prof(PC_POST, 0, 4.0 * rows * N + 4.0 * rows * c.gen_istft_hop_size);
}

static int forward_impl(st2_decoder* d, const float* asr, const float* f0, const float* nn, const float* s,
                        const float* noise, uint64_t seed, float* out, int B, int T, int prec, void* ws,
                        int64_t ws_bytes, cudaStream_t st, bool dry, int64_t* peak_out) {
    const st2_config& c = d->cfg;
    const bool istft = c.variant == 1;
    const bool vocos = c.variant == 4;
    Exec E{d, st, dry, prec, B, (char*)ws, ws_bytes};
    const int spf = d->spf();
    const int S = spf * T, L2 = 2 * T;
    const int up_scale = spf / 2;
    const int C514 = c.dim_in + 2, LD514 = round_up(C514, 64);
    const int C1090 = 1024 + 2 + 64, LD1090 = round_up(C1090, 64);

    float* H = E.allocf((int64_t)B * d->fc_rows);
    E.H = H;
    E.coef = E.allocf((int64_t)B * 2 * 2048);
    float* frames = vocos ? nullptr : E.allocf((int64_t)B * L2 * 9);          // the vocos variant has no harmonic source
    float* har = vocos ? nullptr : E.allocf((int64_t)B * S);
    float* x514 = E.allocf((int64_t)B * T * LD514);
    float* x1090 = E.allocf((int64_t)B * T * LD1090);
    const int C0 = c.upsample_initial_channel;
    float* xg = E.allocf((int64_t)B * 2 * T * C0);
    // per-stage outputs (the mean over the three resblocks), allocated up front
    float* stage_out[4];
    int stage_T[4];
    {
        int Tcur = 2 * T;
        for (int i = 0; i < c.n_stages; ++i) {
            Tcur *= c.upsample_rates[i];
            stage_T[i] = Tcur + ((istft && i + 1 == c.n_stages) ? 1 : 0);
            stage_out[i] = E.allocf((int64_t)B * stage_T[i] * d->stage_channels(i));
        }
    }
    const int har_frames = S / (istft ? c.gen_istft_hop_size : 1) + 1;
    const int HLD = 24;
    float* har22 = istft ? E.allocf((int64_t)B * har_frames * HLD) : nullptr;

    if (E.live()) {
        if (d->profiling) {
            d->prof_recs.clear();
            if (d->prof_events.empty()) {
                cudaEvent_t ev;
                if (cudaEventCreate(&ev) == cudaSuccess) d->prof_events.push_back(ev);
            }
            if (!d->prof_events.empty()) cudaEventRecord(d->prof_events[0], st);
        }
        E.chk(launch_style_fc(s, d->fc_w, d->fc_b, H, B, d->fc_rows, c.style_dim, st));
        E.chk(launch_cf_to_cl(asr, x514, LD514, B, c.dim_in, T, st));
        E.chk(launch_f0n_conv(f0, nn, d->f0_w, d->f0_b, d->n_w, d->n_b, x514, LD514, c.dim_in, C514, x1090, LD1090,
                              1024 + 64, C1090, B, T, st));
        E.prof(PC_MISC, 2.0 * B * d->fc_rows * c.style_dim,
               4.0 * ((double)d->fc_rows * c.style_dim + 2.0 * B * c.dim_in * T + 4.0 * B * L2));
        if (!vocos) {
            E.chk(launch_sinegen_frames(f0, frames, B, L2, up_scale, st));
            E.chk(launch_har_source(f0, frames, noise, seed, d->seed_dev, d->lin_w, d->lin_b, har, B, L2, up_scale, st));
            // SineGen algorithmic bytes (SURVEY.md 8(d)): read 4*B*2T (+ 36*B*S of noise when taped), write 4*B*S
            E.prof(PC_SOURCE, 0, 4.0 * B * L2 + (noise ? 36.0 * B * S : 0.0) + 4.0 * B * S);
        }
        if (istft) {
            E.chk(launch_stft_transform(har, d->stft_fr, d->stft_fi, har22, HLD, B, S, c.gen_istft_n_fft,
                                        c.gen_istft_hop_size, st));
            E.prof(PC_SOURCE, 0, 4.0 * B * S + 4.0 * B * har_frames * (c.gen_istft_n_fft + 2));
        }
    }
    if (!vocos) E.tap("har_source", har, 1, (int64_t)B * S, 1);
    if (istft) E.tap("har", har22, HLD, (int64_t)B * har_frames, c.gen_istft_n_fft + 2);

    // ---- front half: encode, asr_res, decode[0..3] (hifigan.py:461-472)
    E.resblk1d(d->encode, x514, LD514, T, x1090, LD1090);
    {
        const int dt = E.fmt_for("asr_res");
        const bool tc = E.use_tc(d->asr_res, dt);
        const int64_t mark = E.off;
        const void* xin = x514;
        if (tc) {
            void* x16 = E.alloc((int64_t)B * T * LD514 * 2);
            E.norm_act(x514, LD514, T, C514, nullptr, ACT_NONE, 0.f, nullptr, x16, LD514, dt);
            xin = x16;
        }
        E.conv(d->asr_res, xin, LD514, T, tc ? dt : DT_F32, x1090 + 1024, LD1090, T, 1, 0, 1, nullptr, 0, 0, 1.f, 0);
        E.off = mark;
    }
    for (int i = 0; i < 3; ++i) E.resblk1d(d->decode[i], x1090, LD1090, T, x1090, LD1090);
    E.resblk1d(d->decode[3], x1090, LD1090, T, xg, C0);
    E.tap("decode.out", xg, C0, (int64_t)B * 2 * T, C0);
    if (vocos) {
        vocos_generator(E, d, xg, out, 2 * T);
        if (peak_out) *peak_out = E.peak;
        return E.err;
    }

    // ---- generator (hifigan.py:328-345 / istftnet.py:552-573)
    const float* x = xg;
    int Tin = 2 * T;
    int out16 = 0;                                          // the last stage's output is fp16
    for (int i = 0; i < c.n_stages; ++i) {
        const int64_t mark = E.off;
        const int C = d->stage_channels(i), Cin = 2 * C;
        const int u = c.upsample_rates[i], ku = c.upsample_kernel_sizes[i];
        const int Tout = stage_T[i];
        const bool last = (i + 1 == c.n_stages);
        const int shift = (istft && last) ? 1 : 0;          // ReflectionPad1d((1,0))
        const std::string is = std::to_string(i);
        const int dtu = E.fmt_for("generator.ups");
        const int pu = istft ? (ku - u) / 2 : (u / 2 + u % 2);
        const Exec::StagePlan sp = E.plan_stage(i, Tout, E.fused_args(d->ups[i], dtu, Cin, Tin, C, Tout, u, pu, 1, shift));
        const int nc16 = sp.src.x16, xu16 = sp.res[0].x16;
        // x_source = noise_res[i](noise_convs[i](har_source), s)
        float* nc = E.allocf((int64_t)B * Tout * C);
        void* nc16buf = E.alloc((int64_t)B * Tout * C * 2);
        Exec::StatRef nc_stats{nullptr, 0, true};
        bool nc_have_stats = false;
        {
            const ConvW& w = d->noise_convs[i];
            int sf = 1;
            for (int j = i + 1; j < c.n_stages; ++j) sf *= c.upsample_rates[j];
            const int stride = last ? 1 : sf, pad = last ? 0 : (sf + 1) / 2;
            if (istft) {
                E.conv(w, har22, HLD, har_frames, DT_F32, nc, C, Tout, stride, pad, 1, nullptr, 0, 0, 1.f, 0);
            } else {
                // Conv1d(1 -> C) of the harmonic source: dedicated HBM-bound kernel that also emits the InstanceNorm
                // partials of its output (consumed by noise_res[i].adain1[0])
                nc_stats.nparts = noise_conv_parts(Tout, stride);
                void* stp = E.alloc((int64_t)B * nc_stats.nparts * C * 8);
                nc_stats.ptr = stp;
                nc_stats.shift = w.bias;                     // the partials are of the conv without its bias
                nc_have_stats = true;
                if (E.live()) {
                    E.chk(launch_noise_conv(har, w.w32, w.bias, nc16 ? (float*)nc16buf : nc, stp, B, S, Tout, C, w.k, stride, pad, st, nc16));
                    E.prof(PC_SOURCE, 2.0 * B * Tout * C * w.k, 4.0 * B * (double)S + (nc16 ? 2.0 : 4.0) * B * (double)Tout * C);
                }
            }
        }
        E.resblock1(d->noise_res[i], sp.src, nc16 ? (const float*)nc16buf : nc, nc, Tout, nc, nc_have_stats ? &nc_stats : nullptr,
                    nullptr, nc16 ? d->noise_convs[i].bias : nullptr, nc16 ? d->noise_c2b[i] : nullptr);
        // x = ups[i](act(x)) + x_source
        float* xu = E.allocf((int64_t)B * Tout * C);
        Exec::StatRef xu_stats{nullptr, 0, true};
        if (sp.ups_fused) {
            // Snake / LeakyReLU applied on the A-operand path; InstanceNorm statistics of xu from the epilogue
            ConvArgs a = sp.ups;
            xu_stats.nparts = fused_stats_parts(a);
            void* st_xu = E.alloc((int64_t)B * xu_stats.nparts * C * 8);
            xu_stats.ptr = st_xu;
            E.coef_from(Exec::StatRef{nullptr, 0, false}, nullptr, Tin, Cin, Cin);
            a.x = x; a.y = xu; a.res = nc;
            E.conv_fused(a, istft ? ACT_LRELU : ACT_SNAKE, 0.1f, istft ? nullptr : d->gen_alpha[i], st_xu);
        } else {
            const bool tcu = E.use_tc(d->ups[i], dtu);
            void* xs = E.alloc((int64_t)B * Tin * Cin * (tcu ? 2 : 4));
            if (istft) E.norm_act(x, Cin, Tin, Cin, nullptr, ACT_LRELU, 0.1f, nullptr, xs, Cin, tcu ? dtu : DT_F32);
            else E.norm_act(x, Cin, Tin, Cin, nullptr, ACT_SNAKE, 0.f, d->gen_alpha[i], xs, Cin, tcu ? dtu : DT_F32);
            // istftnet: ReflectionPad1d((1,0)) after the last ups = write at row t+1 and mirror row 2 into row 0
            E.conv(d->ups[i], xs, Cin, Tin, tcu ? dtu : DT_F32, xu, C, Tout, u, pu, 1, nc, C, 0, 1.f, 0, shift, shift);
        }
        if (xu16) E.tap16("generator.stage" + is + ".in", xu, (int64_t)B * Tout * C);
        else E.tap("generator.stage" + is + ".in", xu, C, (int64_t)B * Tout, C);
        float* run = E.allocf((int64_t)B * Tout * C);
        void* sum16buf = E.alloc((int64_t)B * Tout * C * 2);
        for (int j = 0; j < c.n_kernels; ++j)
            E.resblock1(d->resblocks[i * c.n_kernels + j], sp.res[j], xu, run, Tout, stage_out[i], sp.ups_fused ? &xu_stats : nullptr,
                        sum16buf);
        out16 = sp.res[c.n_kernels - 1].dest16;
        if (out16) E.tap16("generator.stage" + is + ".out", stage_out[i], (int64_t)B * Tout * C);
        else E.tap("generator.stage" + is + ".out", stage_out[i], C, (int64_t)B * Tout, C);
        x = stage_out[i];
        Tin = Tout;
        E.off = mark;
    }
    const int Cl = d->stage_channels(c.n_stages - 1);
    if (!istft) {
        if (E.live())
            E.chk(launch_post_hifigan(x, Cl, d->gen_alpha[c.n_stages], d->conv_post.w32, d->conv_post.bias, out, B, S, Cl,
                                       prec != ST2_PREC_FP32 ? 1 : 0, st, out16));
        E.prof(PC_POST, 2.0 * B * S * Cl * 7, (out16 ? 2.0 : 4.0) * B * S * Cl + 4.0 * B * S);
    } else {
        const int dt = E.fmt_for("generator.conv_post");
        const bool tc = E.use_tc(d->conv_post, dt);
        void* xa = E.alloc((int64_t)B * Tin * Cl * (tc ? 2 : 4));
        E.norm_act(x, Cl, Tin, Cl, nullptr, ACT_LRELU, 0.01f, nullptr, xa, Cl, tc ? dt : DT_F32);
        float* y22 = E.allocf((int64_t)B * Tin * HLD);
        E.conv(d->conv_post, xa, Cl, Tin, tc ? dt : DT_F32, y22, HLD, Tin, 1, 3, 1, nullptr, 0, 0, 1.f, 0);
        E.tap("generator.conv_post", y22, HLD, (int64_t)B * Tin, c.gen_istft_n_fft + 2);
        if (E.live())
            E.chk(launch_istft_head(y22, HLD, d->stft_br, d->stft_bi, out, B, Tin, S, c.gen_istft_n_fft,
                                    c.gen_istft_hop_size, st));
        E.prof(PC_POST, 0, 4.0 * B * Tin * (c.gen_istft_n_fft + 2) + 4.0 * B * S);
    }
    if (peak_out) *peak_out = E.peak;
    return E.err;
}

// ---- process-wide tuning switches (common.cuh)
namespace {
struct TuneField { const char* name; int Tune::*field; };
const TuneField kTuneFields[] = {
    {"no_pipe", &Tune::no_pipe}, {"row_always", &Tune::row_always}, {"row_sub", &Tune::row_sub},
    {"no_row_inline_coef", &Tune::no_row_inline_coef}, {"verbose", &Tune::verbose}};
Tune& tune_storage() {
    static Tune t;
    return t;
}
}  // namespace
const Tune& tune() { return tune_storage(); }
int tune_set(const char* name, int value) {
    for (const TuneField& f : kTuneFields)
        if (strcmp(name, f.name) == 0) {
            tune_storage().*(f.field) = value;
            return ST2_OK;
        }
    set_error("set_tuning: unknown switch '%s'", name);
    return ST2_ERR_INVALID;
}
int device_num_sms() {
    static int sms[kMaxDevices] = {};
    const int dev = current_device_slot();
    if (sms[dev] == 0) {
        int v = 0;
        cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
        sms[dev] = v > 0 ? v : 148;
    }
    return sms[dev];
}

}  // namespace st2

// ------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------
extern "C" {

int st2_abi_version(void) { return ST2_ABI_VERSION; }
const char* st2_last_error(void) { return st2::g_err; }

static int create_handle(const st2_config* cfg, st2_decoder** out) {
    st2_decoder* d = new (std::nothrow) st2_decoder();
    ST2_REQUIRE(d != nullptr, "create: out of memory");
    d->cfg = *cfg;
    int dev = 0;
    cudaDeviceProp prop;
    if (cudaGetDevice(&dev) == cudaSuccess && cudaGetDeviceProperties(&prop, dev) == cudaSuccess)
        d->tc_ok = (prop.major == 10);
    *out = d;
    return ST2_OK;
}

int st2_decoder_create(const st2_config* cfg, st2_decoder** out) {
    ST2_REQUIRE(cfg != nullptr && out != nullptr, "create: null argument");
    ST2_REQUIRE(cfg->variant == 0 || cfg->variant == 1 || cfg->variant == 4,
                "create: variant must be 0 (hifigan), 1 (istftnet) or 4 (vocos)");
    ST2_REQUIRE(cfg->dim_in == 512 && cfg->style_dim >= 4 && cfg->style_dim <= 1024, "create: dim_in must be 512");
    if (cfg->variant == 4) {
        // Modules/vocos.py:364-393: decode.3 ends at 512 channels = the generator's dim; ISTFT 'same' padding (vocos.py:203)
        ST2_REQUIRE(cfg->upsample_initial_channel == 512 && cfg->n_stages == 0, "create: vocos has no upsampling stages");
        ST2_REQUIRE(cfg->num_layers >= 1 && cfg->num_layers <= 16 && cfg->intermediate_dim >= 64 && cfg->intermediate_dim <= 2048 &&
                        cfg->intermediate_dim % 64 == 0,
                    "create: vocos needs 1..16 layers and an intermediate_dim that is a multiple of 64, at most 2048");
        ST2_REQUIRE(cfg->gen_istft_hop_size >= 1 && cfg->gen_istft_n_fft % 16 == 0 && cfg->gen_istft_n_fft >= cfg->gen_istft_hop_size &&
                        (cfg->gen_istft_n_fft - cfg->gen_istft_hop_size) % 2 == 0 && cfg->gen_istft_n_fft <= 4096,
                    "create: vocos ISTFT needs n_fft a multiple of 16 (<= 4096), hop <= n_fft, n_fft - hop even");
        return create_handle(cfg, out);
    }
    ST2_REQUIRE(cfg->n_stages >= 1 && cfg->n_stages <= 4 && cfg->n_kernels == 3, "create: unsupported stage/kernel count");
    ST2_REQUIRE(cfg->upsample_initial_channel % 64 == 0 && (cfg->upsample_initial_channel >> cfg->n_stages) >= 4 &&
                    ((cfg->upsample_initial_channel >> cfg->n_stages) % 4) == 0,
                "create: unsupported upsample_initial_channel");
    // the AdaIN coefficient buffer of a forward holds 2 x 2048 floats per utterance (Exec::coef)
    ST2_REQUIRE(cfg->upsample_initial_channel <= 2048, "create: upsample_initial_channel must be <= 2048");
    for (int i = 0; i < cfg->n_stages; ++i)
        ST2_REQUIRE(cfg->upsample_rates[i] >= 1 && cfg->upsample_kernel_sizes[i] % cfg->upsample_rates[i] == 0,
                    "create: upsample kernel must be a multiple of its rate");
    if (cfg->variant == 1)
        ST2_REQUIRE(cfg->gen_istft_n_fft == 20 && cfg->gen_istft_hop_size == 5, "create: iSTFT head supports n_fft=20, hop=5");
    return create_handle(cfg, out);
}

void st2_decoder_destroy(st2_decoder* d) {
    if (!d) return;
    for (void* p : d->allocs) cudaFree(p);
    for (cudaEvent_t ev : d->prof_events) cudaEventDestroy(ev);
    delete d;
}

int st2_decoder_set_weight(st2_decoder* d, const char* name, const float* dev_ptr, const int64_t* shape, int32_t ndim) {
    ST2_REQUIRE(d && name && dev_ptr && (shape || ndim == 0) && ndim >= 0 && ndim <= 4, "set_weight: bad argument");
    st2::RawTensor t;
    t.ptr = dev_ptr;
    for (int i = 0; i < ndim; ++i) t.shape.push_back(shape[i]);
    d->raw[name] = t;
    return ST2_OK;
}

int st2_decoder_finalize(st2_decoder* d, void* stream) {
    ST2_REQUIRE(d != nullptr, "finalize: null handle");
    for (void* p : d->allocs) cudaFree(p);
    d->allocs.clear();
    d->finalized = false;
    int e = st2::finalize_impl(d, (cudaStream_t)stream);
    if (e != ST2_OK) {
        for (void* p : d->allocs) cudaFree(p);
        d->allocs.clear();
    }
    return e;
}

int64_t st2_decoder_num_params(const st2_decoder* d) { return d ? d->num_params : 0; }

int64_t st2_decoder_workspace_bytes(const st2_decoder* d, int32_t B, int32_t T, int32_t precision) {
    if (!d || !d->finalized || d->cfg.variant == 2 || d->cfg.variant == 3 || B <= 0 || T <= 0) {
        st2::set_error("workspace_bytes: handle not finalized (or a predictor handle) or bad shape");
        return ST2_ERR_STATE;
    }
    int64_t peak = 0;
    int e = st2::forward_impl(const_cast<st2_decoder*>(d), nullptr, nullptr, nullptr, nullptr, nullptr, 0, nullptr, B, T,
                              precision, nullptr, 0, nullptr, true, &peak);
    if (e != ST2_OK) return e;
    return peak + 256;
}

int st2_decoder_forward(st2_decoder* d, const float* asr, const float* f0, const float* n, const float* s,
                        const float* noise, uint64_t seed, float* out, int32_t B, int32_t T, int32_t precision,
                        void* workspace, int64_t workspace_bytes, void* stream) {
    ST2_REQUIRE(d != nullptr, "forward: null handle");
    if (!d->finalized || d->cfg.variant == 2 || d->cfg.variant == 3) {
        st2::set_error("forward: st2_decoder_finalize has not been called (or this is a predictor / text-encoder handle)");
        return ST2_ERR_STATE;
    }
    ST2_REQUIRE(asr && f0 && n && s && out && workspace, "forward: null tensor");
    ST2_REQUIRE(B > 0 && T >= 2, "forward: need B>0 and T>=2 (got B=%d T=%d)", B, T);
    ST2_REQUIRE(precision >= ST2_PREC_FP32 && precision <= ST2_PREC_FP16, "forward: bad precision %d", precision);
    if (precision != ST2_PREC_FP32 && !d->tc_ok) {
        st2::set_error("forward: tensor-core precision requires an sm_100 device");
        return ST2_ERR_UNSUPPORTED;
    }
    ST2_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "forward: workspace must be 256-byte aligned");
    st2::g_launch_count = 0;
    int e = st2::forward_impl(d, asr, f0, n, s, noise, seed, out, B, T, precision, workspace, workspace_bytes,
                              (cudaStream_t)stream, false, nullptr);
    d->last_launches = st2::g_launch_count;
    return e;
}

int st2_decoder_set_tap(st2_decoder* d, const char* name, float* dst, int64_t capacity) {
    ST2_REQUIRE(d && name, "set_tap: bad argument");
    if (dst == nullptr) d->taps.erase(name);
    else d->taps[name] = st2::Tap{dst, capacity};
    return ST2_OK;
}

int st2_decoder_set_option(st2_decoder* d, const char* name, int32_t value) {
    ST2_REQUIRE(d && name, "set_option: bad argument");
    struct { const char* n; int* v; } opts[] = {{"fp16_storage", &d->fp16_storage}, {"fp16_xt", &d->opt_xt16}, {"fp16_run", &d->opt_run16},
                                                {"fp16_xu", &d->opt_xu16}, {"fp16_sum", &d->opt_sum16},
                                                {"fp16_src", &d->opt_src16}, {"fp16_out", &d->opt_out16}};
    for (auto& o : opts)
        if (strcmp(name, o.n) == 0) {
            *o.v = value ? 1 : 0;
            return ST2_OK;
        }
    st2::set_error("set_option: unknown option '%s'", name);
    return ST2_ERR_INVALID;
}

int st2_set_tuning(const char* name, int32_t value) {
    ST2_REQUIRE(name != nullptr, "set_tuning: null name");
    return st2::tune_set(name, value);
}

int st2_decoder_set_seed_buffer(st2_decoder* d, const uint64_t* dev_seed) {
    ST2_REQUIRE(d != nullptr, "set_seed_buffer: null handle");
    d->seed_dev = dev_seed;
    return ST2_OK;
}

int64_t st2_decoder_last_launch_count(const st2_decoder* d) { return d ? d->last_launches : 0; }

int st2_decoder_set_profiling(st2_decoder* d, int32_t enable) {
    ST2_REQUIRE(d != nullptr, "set_profiling: null handle");
    d->profiling = enable != 0;
    d->prof_recs.clear();
    return ST2_OK;
}

int st2_profile_num_categories(void) { return st2::PC_COUNT; }

const char* st2_profile_category_name(int32_t cat) {
    static const char* names[st2::PC_COUNT] = {"conv_tc", "conv_simt", "norm_stats", "norm_coef", "affine_act",
                                               "source", "post", "misc", "conv_fused", "conv_pipe", "lstm", "conv_row"};
    return (cat >= 0 && cat < st2::PC_COUNT) ? names[cat] : "";
}

int64_t st2_decoder_get_profile_launches(st2_decoder* d, int64_t max_n, int32_t* cat, float* ms, double* flops,
                                         double* bytes) {
    if (!d || !cat || !ms || !flops || !bytes) { st2::set_error("get_profile_launches: null argument"); return ST2_ERR_INVALID; }
    const size_t n = d->prof_recs.size();
    if (n == 0) return 0;
    if (d->prof_events.size() <= n) { st2::set_error("get_profile_launches: event pool inconsistent"); return ST2_ERR_STATE; }
    ST2_CUDA_CHECK(cudaEventSynchronize(d->prof_events[n]));
    const size_t m = n < (size_t)max_n ? n : (size_t)max_n;
    for (size_t i = 0; i < m; ++i) {
        float t = 0.f;
        ST2_CUDA_CHECK(cudaEventElapsedTime(&t, d->prof_events[i], d->prof_events[i + 1]));
        cat[i] = d->prof_recs[i].cat; ms[i] = t; flops[i] = d->prof_recs[i].flops; bytes[i] = d->prof_recs[i].bytes;
    }
    return (int64_t)m;
}

int st2_decoder_get_profile(st2_decoder* d, double* ms, int64_t* launches, double* flops, double* bytes) {
    ST2_REQUIRE(d && ms && launches && flops && bytes, "get_profile: null argument");
    for (int i = 0; i < st2::PC_COUNT; ++i) { ms[i] = 0; launches[i] = 0; flops[i] = 0; bytes[i] = 0; }
    const size_t n = d->prof_recs.size();
    if (n == 0) return ST2_OK;
    ST2_REQUIRE(d->prof_events.size() > n, "get_profile: event pool inconsistent");
    ST2_CUDA_CHECK(cudaEventSynchronize(d->prof_events[n]));
    for (size_t i = 0; i < n; ++i) {
        float t = 0.f;
        ST2_CUDA_CHECK(cudaEventElapsedTime(&t, d->prof_events[i], d->prof_events[i + 1]));
        const auto& r = d->prof_recs[i];
        ms[r.cat] += t;
        launches[r.cat] += 1;
        flops[r.cat] += r.flops;
        bytes[r.cat] += r.bytes;
    }
    return ST2_OK;
}

}  // extern "C"
