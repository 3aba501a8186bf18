// Shared by decoder.cu and predictor.cu: the opaque handle behind include/st2_b200.h, the load-time weight Packer and the
// forward-program executor Exec (workspace carving, per-launch profile, the AdainResBlk1d / AdaINResBlock1 block programs
// and the conv dispatch).  Header-only on purpose: both translation units run the same block programs.
#pragma once
#include <stdlib.h>
#include <string.h>

#include <map>
#include <new>
#include <string>
#include <vector>

#include "common.cuh"

namespace st2 {

extern thread_local char g_err[1024];

struct RawTensor {
    const float* ptr;
    std::vector<int64_t> shape;
    int64_t numel() const {
        int64_t n = 1;
        for (auto s : shape) n *= s;
        return n;
    }
};

struct ConvW {
    float* w32 = nullptr;       // [k][Cin][Cout]
    void* w16[3] = {nullptr, nullptr, nullptr};   // index by OutDtype: [k][CoutPad][CinPad]
    float* bias = nullptr;
    int Cin = 0, Cout = 0, k = 0;
    int cin_pad = 0, cout_pad = 0;
    bool transposed = false;
};

struct AdaINRef { int h_off = 0; int C = 0; };

struct ResBlock1W {           // AdaINResBlock1 (hifigan.py:26-74)
    ConvW c1[3], c2[3];
    AdaINRef n1[3], n2[3];
    float* alpha1[3] = {nullptr, nullptr, nullptr};
    float* alpha2[3] = {nullptr, nullptr, nullptr};
    int k = 0, C = 0;
    int dil[3] = {1, 3, 5};
    std::string name;
};

struct ResBlk1dW {            // AdainResBlk1d (hifigan.py:359-403)
    ConvW conv1, conv2, conv1x1;
    bool has_sc = false, upsample = false;
    AdaINRef norm1, norm2;
    float* pool_w = nullptr;  // [3][ld_in]
    float* pool_b = nullptr;  // [ld_in]
    int Cin = 0, Cout = 0;
    std::string name;
};

struct LstmW {                // bidirectional nn.LSTM(I, H): input half as two 1x1 convs, W_hh^T / b_hh for the recurrence kernel
    ConvW ih[2];
    float* whh = nullptr;     // [2][H][4H]
    float* bhh = nullptr;     // [2][4H]
};

struct Tap { float* dst; int64_t cap; };

}  // namespace st2

using namespace st2;

struct st2_decoder {
    st2_config cfg;
    std::map<std::string, RawTensor> raw;
    bool finalized = false;
    std::vector<void*> allocs;
    int64_t num_params = 0;
    int64_t last_launches = 0;
    const uint64_t* seed_dev = nullptr;     // optional device-resident Philox seed (st2_decoder_set_seed_buffer)
    bool tc_ok = false;
    // st2_decoder_set_option("fp16_storage"): stage-private tensors of the 16-bit paths in fp16, and each kind alone ("fp16_xt",
    // "fp16_run", "fp16_xu", "fp16_sum", "fp16_src", "fp16_out"); read by Exec::plan_stage only
    int fp16_storage = 1;
    int opt_xt16 = 1, opt_run16 = 1, opt_xu16 = 1, opt_sum16 = 1, opt_src16 = 1, opt_out16 = 1;

    ResBlk1dW encode, decode[4];
    float *f0_w = nullptr, *f0_b = nullptr, *n_w = nullptr, *n_b = nullptr;
    ConvW asr_res;
    float *lin_w = nullptr, *lin_b = nullptr;
    float* gen_alpha[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    ConvW noise_convs[4], ups[4], conv_post;
    ResBlock1W noise_res[4], resblocks[12];
    float *fc_w = nullptr, *fc_b = nullptr;
    int fc_rows = 0;
    float *stft_fr = nullptr, *stft_fi = nullptr, *stft_br = nullptr, *stft_bi = nullptr;
    std::map<std::string, Tap> taps;

    // variant 4: Vocos generator (Modules/vocos.py:103-162, :235-296): ConvNeXt blocks, final LayerNorm, ISTFTHead
    struct ConvNeXtW { float* dw_w = nullptr; float* dw_b = nullptr; AdaINRef norm; ConvW pw1, pw2; };
    ConvNeXtW vx[16];
    float* noise_c2b[4] = {nullptr, nullptr, nullptr, nullptr};   // noise_res[i].convs2.0.bias + noise_convs[i].bias (fp16_src path)
    float* vx_ln = nullptr;                 // final_layer_norm weight[dim] | bias[dim]
    ConvW vx_out;                           // ISTFTHead.out, columns padded to vx_kpad
    ConvW vx_basis;                         // windowed inverse real DFT as a [vx_kpad, n_fft] matrix (vocos.cu)
    float* vx_window = nullptr;             // generator.stft.istft.window [n_fft]
    int vx_kpad = 0;

    // variant 2: the F0 / energy predictor ProsodyPredictor.F0Ntrain (models.py:407-419, :448-461); cfg.dim_in = d_hid
    LstmW shared;                           // models.py:407
    // duration half (row N2; packed only when the caller handed its weights over): DurationEncoder (models.py:468-483),
    // `lstm` (models.py:404), `duration_proj` (models.py:405)
    bool has_duration = false;
    int dur_layers = 0;
    LstmW enc_lstm[4];
    AdaINRef enc_norm[4];                   // AdaLayerNorm fc rows (gamma(C) | beta(C)) in the shared style matrix
    LstmW dur_lstm;
    float *dur_w = nullptr, *dur_b = nullptr;   // duration_proj.linear_layer [max_dur][d_hid], [max_dur]
    int max_dur = 0;

    // variant 3: TextEncoder (models.py:238-285); cfg.dim_in = channels
    int te_depth = 0, te_kernel = 0, te_symbols = 0;
    float* te_embedding = nullptr;          // [n_symbols][channels]
    ConvW te_conv[8];
    float* te_gamma[8] = {};                // gamma[c] followed by beta[c]
    LstmW te_lstm;
    ResBlk1dW pred_blk[2][3];               // F0.{0,1,2}, N.{0,1,2}
    ConvW pred_proj[2];                     // F0_proj, N_proj

    // per-launch event profile (one boundary event after every launch of a profiled forward)
    struct ProfRec { int cat; double flops; double bytes; };
    bool profiling = false;
    std::vector<cudaEvent_t> prof_events;
    std::vector<ProfRec> prof_recs;

    int spf() const {    // samples per asr frame
        int p = 2;
        for (int i = 0; i < cfg.n_stages; ++i) p *= cfg.upsample_rates[i];
        return p * ((cfg.variant == 1 || cfg.variant == 4) ? cfg.gen_istft_hop_size : 1);
    }
    int stage_channels(int i) const { return cfg.upsample_initial_channel >> (i + 1); }
};

namespace st2 {

static inline int round_up(int v, int m) { return (v + m - 1) / m * m; }

// ------------------------------------------------------------------------------------------
// load time
// ------------------------------------------------------------------------------------------
struct Packer {
    st2_decoder* d;
    cudaStream_t st;
    int err = ST2_OK;
    std::vector<std::pair<std::string, int>> adain_list;   // (prefix, C) in h_off order

    void* dalloc(size_t bytes) {
        void* p = nullptr;
        if (cudaMalloc(&p, bytes ? bytes : 4) != cudaSuccess) {
            set_error("cudaMalloc(%zu) failed while packing weights", bytes);
            err = ST2_ERR_CUDA;
            return nullptr;
        }
        d->allocs.push_back(p);
        return p;
    }
    const RawTensor* get(const std::string& n, bool required = true) {
        auto it = d->raw.find(n);
        if (it == d->raw.end()) {
            if (required && err == ST2_OK) {
                set_error("missing weight '%s'", n.c_str());
                err = ST2_ERR_INVALID;
            }
            return nullptr;
        }
        return &it->second;
    }
    float* copy(const std::string& n, int64_t expect_numel) {
        const RawTensor* t = get(n);
        if (!t) return nullptr;
        if (t->numel() != expect_numel) {
            set_error("weight '%s' has %lld elements, expected %lld", n.c_str(), (long long)t->numel(),
                      (long long)expect_numel);
            err = ST2_ERR_INVALID;
            return nullptr;
        }
        float* p = (float*)dalloc(expect_numel * sizeof(float));
        if (p && cudaMemcpyAsync(p, t->ptr, expect_numel * sizeof(float), cudaMemcpyDeviceToDevice, st) != cudaSuccess)
            err = ST2_ERR_CUDA;
        return p;
    }
    void conv(ConvW& c, const std::string& n, int Cin, int Cout, int k, bool transposed, bool bias, bool want16) {
        c.Cin = Cin; c.Cout = Cout; c.k = k; c.transposed = transposed;
        // legacy weight_norm keys (hifigan.py / istftnet.py), the parametrizations ones of Modules/vocos.py:10, or a plain weight
        const RawTensor* g = get(n + ".weight_g", false);
        const RawTensor* v = nullptr;
        if (g) {
            v = get(n + ".weight_v");
        } else if ((g = get(n + ".parametrizations.weight.original0", false)) != nullptr) {
            v = get(n + ".parametrizations.weight.original1");
        } else {
            v = get(n + ".weight");
        }
        if (!v) return;
        const int d0 = transposed ? Cin : Cout, d1 = transposed ? Cout : Cin;
        if (v->shape.size() != 3 || v->shape[0] != d0 || v->shape[1] != d1 || v->shape[2] != k ||
            (g && g->numel() != d0)) {
            set_error("weight '%s' has the wrong shape (expected [%d,%d,%d])", n.c_str(), d0, d1, k);
            err = ST2_ERR_INVALID;
            return;
        }
        c.w32 = (float*)dalloc((size_t)k * Cin * Cout * sizeof(float));
        if (!c.w32) return;
        if (launch_fold_pack(g ? g->ptr : nullptr, v->ptr, c.w32, d0, d1, k, transposed ? 1 : 0, st) != ST2_OK)
            err = ST2_ERR_CUDA;
        if (bias) c.bias = copy(n + ".bias", Cout);
        if (want16 && d->tc_ok) {
            c.cin_pad = round_up(Cin, 64);
            c.cout_pad = round_up(Cout, 16);
            for (int dt = DT_BF16; dt <= DT_F16; ++dt) {
                c.w16[dt] = dalloc((size_t)k * c.cin_pad * c.cout_pad * 2);
                if (c.w16[dt] &&
                    launch_pack_w16(c.w32, c.w16[dt], k, Cin, Cout, c.cin_pad, c.cout_pad, dt, st) != ST2_OK)
                    err = ST2_ERR_CUDA;
            }
        }
    }
    // nn.Linear / nn.LSTM input matrix [Cout, Cin] as a 1x1 conv (packed [1][Cin][Cout] + 16-bit copies)
    // col_scale (optional, [Cout]): every output column and the bias are multiplied by it (a per-channel layer scale folded in);
    // cout_pad > Cout: zero weight columns / zero bias entries up to cout_pad, which becomes the layer's Cout
    void linear(ConvW& c, const std::string& wname, const std::string& bname, int Cin, int Cout, const float* col_scale = nullptr,
                int cout_pad = 0) {
        const int Cp = cout_pad > Cout ? cout_pad : Cout;
        c.Cin = Cin; c.Cout = Cp; c.k = 1; c.transposed = false;
        const RawTensor* v = get(wname);
        if (!v) return;
        if (v->numel() != (int64_t)Cin * Cout || v->shape.empty() || v->shape[0] != Cout) {
            set_error("weight '%s' has the wrong shape (expected [%d,%d])", wname.c_str(), Cout, Cin);
            err = ST2_ERR_INVALID;
            return;
        }
        c.w32 = (float*)dalloc((size_t)Cin * Cp * sizeof(float));
        if (!c.w32) return;
        if (Cp == Cout) {
            if (launch_fold_pack(nullptr, v->ptr, c.w32, Cout, Cin, 1, 0, st) != ST2_OK) err = ST2_ERR_CUDA;
        } else {
            float* tmp = (float*)dalloc((size_t)Cin * Cout * sizeof(float));
            if (!tmp) return;
            if (launch_fold_pack(nullptr, v->ptr, tmp, Cout, Cin, 1, 0, st) != ST2_OK) err = ST2_ERR_CUDA;
            if (cudaMemsetAsync(c.w32, 0, (size_t)Cin * Cp * sizeof(float), st) != cudaSuccess ||
                cudaMemcpy2DAsync(c.w32, (size_t)Cp * sizeof(float), tmp, (size_t)Cout * sizeof(float), (size_t)Cout * sizeof(float),
                                  Cin, cudaMemcpyDeviceToDevice, st) != cudaSuccess)
                err = ST2_ERR_CUDA;
        }
        if (!bname.empty()) {
            const float* b = copy(bname, Cout);
            c.bias = (float*)dalloc((size_t)Cp * sizeof(float));
            if (!b || !c.bias) return;
            if (cudaMemsetAsync(c.bias, 0, (size_t)Cp * sizeof(float), st) != cudaSuccess ||
                cudaMemcpyAsync(c.bias, b, (size_t)Cout * sizeof(float), cudaMemcpyDeviceToDevice, st) != cudaSuccess)
                err = ST2_ERR_CUDA;
        }
        if (col_scale && launch_scale_cols(c.w32, c.bias, Cin, Cp, Cout, col_scale, st) != ST2_OK) err = ST2_ERR_CUDA;
        if (d->tc_ok && Cin % 64 == 0 && Cp % 16 == 0) {
            c.cin_pad = Cin; c.cout_pad = Cp;
            for (int dt = DT_BF16; dt <= DT_F16; ++dt) {
                c.w16[dt] = dalloc((size_t)Cin * Cp * 2);
                if (c.w16[dt] && launch_pack_w16(c.w32, c.w16[dt], 1, Cin, Cp, Cin, Cp, dt, st) != ST2_OK) err = ST2_ERR_CUDA;
            }
        }
    }
    void adain(AdaINRef& a, const std::string& prefix, int C) {
        a.C = C;
        a.h_off = d->fc_rows;
        d->fc_rows += 2 * C;
        adain_list.push_back({prefix, C});
    }
    void resblk1d(ResBlk1dW& b, const std::string& n, int Cin, int Cout, bool upsample) {
        b.name = n; b.Cin = Cin; b.Cout = Cout; b.upsample = upsample; b.has_sc = (Cin != Cout);
        conv(b.conv1, n + ".conv1", Cin, Cout, 3, false, true, true);
        conv(b.conv2, n + ".conv2", Cout, Cout, 3, false, true, true);
        if (b.has_sc) conv(b.conv1x1, n + ".conv1x1", Cin, Cout, 1, false, false, true);
        adain(b.norm1, n + ".norm1", Cin);
        adain(b.norm2, n + ".norm2", Cout);
        if (upsample) {
            // depthwise ConvTranspose1d weight [C,1,3] -> [3][ld] (zero padded), bias [ld]
            const int ld = round_up(Cin, 64);
            ConvW tmp;
            conv(tmp, n + ".pool", Cin, 1, 3, true, false, false);
            tmp.bias = copy(n + ".pool.bias", Cin);
            b.pool_w = (float*)dalloc((size_t)3 * ld * sizeof(float));
            b.pool_b = (float*)dalloc((size_t)ld * sizeof(float));
            if (err != ST2_OK || !b.pool_w || !b.pool_b) return;
            cudaMemsetAsync(b.pool_w, 0, (size_t)3 * ld * sizeof(float), st);
            cudaMemsetAsync(b.pool_b, 0, (size_t)ld * sizeof(float), st);
            cudaMemcpy2DAsync(b.pool_w, (size_t)ld * sizeof(float), tmp.w32, (size_t)Cin * sizeof(float),
                              (size_t)Cin * sizeof(float), 3, cudaMemcpyDeviceToDevice, st);
            cudaMemcpyAsync(b.pool_b, tmp.bias, (size_t)Cin * sizeof(float), cudaMemcpyDeviceToDevice, st);
        }
    }
    void resblock1(ResBlock1W& b, const std::string& n, int C, int k, const int* dil) {
        b.name = n; b.C = C; b.k = k;
        for (int j = 0; j < 3; ++j) {
            b.dil[j] = dil[j];
            const std::string js = std::to_string(j);
            conv(b.c1[j], n + ".convs1." + js, C, C, k, false, true, true);
            conv(b.c2[j], n + ".convs2." + js, C, C, k, false, true, true);
            adain(b.n1[j], n + ".adain1." + js, C);
            adain(b.n2[j], n + ".adain2." + js, C);
            b.alpha1[j] = copy(n + ".alpha1." + js, C);
            b.alpha2[j] = copy(n + ".alpha2." + js, C);
        }
    }
};

// one bidirectional nn.LSTM: W_ih as 1x1 convs (+ b_ih), W_hh transposed for the recurrence kernel
// one bidirectional nn.LSTM / ProsodyPredictor / TextEncoder weights (predictor.cu); Decoder weights (decoder.cu)
void pack_predictor(st2_decoder* d, Packer& P);
void pack_text_encoder(st2_decoder* d, Packer& P);

// ------------------------------------------------------------------------------------------
// forward program
// ------------------------------------------------------------------------------------------
struct Exec {
    st2_decoder* d;
    cudaStream_t st;
    bool dry;                 // plan only: compute the workspace high-water mark
    int prec;                 // st2_precision
    int B;
    char* base;
    int64_t cap, off = 0, peak = 0;
    int err = ST2_OK;
    const float* H = nullptr; // style rows [B][fc_rows]
    float* coef = nullptr;    // [B][2][2048]
    int coef_ld = 0;          // stride the last coefficient kernel wrote with
    const int32_t* lengths = nullptr;   // ragged token batches of the text modules (device, [B]); nullptr = equal lengths

    void* alloc(int64_t bytes) {
        off = (off + 255) / 256 * 256;
        void* p = dry ? nullptr : base + off;
        off += bytes;
        if (off > peak) peak = off;
        if (!dry && off > cap && err == ST2_OK) {
            set_error("workspace too small: need at least %lld bytes, have %lld", (long long)off, (long long)cap);
            err = ST2_ERR_WORKSPACE;
        }
        return p;
    }
    float* allocf(int64_t n) { return (float*)alloc(n * (int64_t)sizeof(float)); }
    bool live() const { return !dry && err == ST2_OK; }
    void chk(int e) { if (e != ST2_OK && err == ST2_OK) err = e; }

    // boundary event after the launch(es) just issued; flops / bytes are the ALGORITHMIC figures
    void prof(int cat, double flops, double bytes) {
        if (!d->profiling || !live()) return;
        const size_t idx = d->prof_recs.size() + 1;      // event 0 = start of the forward
        while (d->prof_events.size() <= idx) {
            cudaEvent_t ev;
            if (cudaEventCreate(&ev) != cudaSuccess) { chk(ST2_ERR_CUDA); return; }
            d->prof_events.push_back(ev);
        }
        cudaEventRecord(d->prof_events[idx], st);
        d->prof_recs.push_back({cat, flops, bytes});
    }

    int fmt_for(const std::string& name) const {
        if (prec == ST2_PREC_FP32) return DT_F32;
        if (prec == ST2_PREC_FP16) return DT_F16;
        if (d->cfg.variant == 2 || d->cfg.variant == 3) return DT_F16;   // predictor / text encoder: 0.4 % of the decoder's FLOPs, its outputs steer the SineGen phase
        // bf16 for the generator resblocks / ups (96 % of the FLOPs).  fp16 operands (same tensor
        // throughput) for generator.noise_res -- bf16 there alone costs ~9 dB of SNR -- and for the
        // front half (encode / decode / asr_res, K up to 3270), whose five chained blocks otherwise
        // reach 1.2e-2 per-layer relative L2 (DESIGN.md, precision study).
        if (name.find("noise_res") != std::string::npos || name.find("encode") != std::string::npos ||
            name.find("decode") != std::string::npos || name.find("asr_res") != std::string::npos)
            return DT_F16;
        return DT_BF16;
    }

    void tap(const std::string& name, const float* src, int ld, int64_t rows, int C) {
        if (!live()) return;
        auto it = d->taps.find(name);
        if (it == d->taps.end() || it->second.dst == nullptr) return;
        if (rows * C > it->second.cap) {
            set_error("tap '%s' needs %lld floats, buffer has %lld", name.c_str(), (long long)(rows * C),
                      (long long)it->second.cap);
            err = ST2_ERR_INVALID;
            return;
        }
        chk(launch_copy_dense(src, ld, it->second.dst, rows, C, st));
        prof(PC_MISC, 0, 8.0 * rows * C);
    }

    // tap of a dense fp16 tensor (the intra-block tensor of the fused resblocks)
    void tap16(const std::string& name, const void* src, int64_t n) {
        if (!live()) return;
        auto it = d->taps.find(name);
        if (it == d->taps.end() || it->second.dst == nullptr) return;
        if (n > it->second.cap) {
            set_error("tap '%s' needs %lld floats, buffer has %lld", name.c_str(), (long long)n, (long long)it->second.cap);
            err = ST2_ERR_INVALID;
            return;
        }
        chk(launch_half_to_float(src, it->second.dst, n, st));
        prof(PC_MISC, 0, 6.0 * n);
    }

    // y = act(AdaIN(x)) or act(x) when `n` is null.  x fp32 [B,T,ld_x]; y dtype dt, pitch ld_y.
    void norm_act(const float* x, int ld_x, int T, int C, const AdaINRef* n, int act, float slope, const float* alpha,
                  void* y, int ld_y, int dt) {
        const int Cpad = ld_y < ld_x ? ld_y : ld_x;
        if (Cpad > 2048 && err == ST2_OK) {
            set_error("coefficient buffer holds 2048 channels, layer needs %d", Cpad);
            err = ST2_ERR_UNSUPPORTED;
        }
        void* scratch = nullptr;
        const int64_t mark = off;
        if (n) scratch = alloc(adain_scratch_bytes(B, T, C));
        if (live()) {
            const double numel = (double)B * T * C;
            if (n) {
                chk(launch_in_stats(x, ld_x, B, T, C, scratch, st));
                prof(PC_NORM_STATS, 0, numel * 4);
            }
            if (err == ST2_OK) chk(launch_adain_coef(scratch, n ? H : nullptr, d->fc_rows, n ? n->h_off : 0, coef, B, T, C, Cpad, st));
            prof(PC_NORM_COEF, 0, 0);
            if (err == ST2_OK) chk(launch_affine_act(x, ld_x, coef, alpha, act, slope, y, ld_y, dt, B, T, Cpad, st));
            prof(PC_AFFINE_ACT, 0, numel * (4 + (dt == DT_F32 ? 4 : 2)));
        }
        off = mark;
    }

    bool use_tc(const ConvW& w, int dt) const { return dt != DT_F32 && w.w16[dt] != nullptr; }

    // geometry of Conv1d / (polyphase) ConvTranspose1d in the common ConvArgs contract
    bool fill_args(ConvArgs& a, const ConvW& w, int Tin, int Tout, int stride, int padding, int dilation, int out_row_shift) {
        memset(&a, 0, sizeof(a));
        a.B = B; a.Cin = w.Cin; a.Cout = w.Cout;
        a.Tin = Tin; a.Tout = Tout;
        a.w = w.w32; a.bias = w.bias;
        if (!w.transposed) {
            a.M = Tout; a.ntaps = w.k; a.tap_step = dilation; a.in_off = -padding; a.in_stride = stride;
            a.phases = 1; a.w_step = 1; a.out_stride = 1; a.out_pad = -out_row_shift;
        } else {
            if (w.k % stride != 0) {
                set_error("ConvTranspose1d k=%d must be a multiple of stride=%d", w.k, stride);
                err = ST2_ERR_UNSUPPORTED;
                return false;
            }
            a.ntaps = w.k / stride; a.tap_step = -1; a.in_off = 0; a.in_stride = 1;
            a.phases = stride; a.w_step = stride; a.out_stride = stride; a.out_pad = padding - out_row_shift;
            a.M = (Tout - 1 - out_row_shift + padding) / stride + 1;
        }
        return true;
    }

    // Conv1d (stride 1 here except noise_convs) / ConvTranspose1d through the common ConvArgs contract
    void conv(const ConvW& w, const void* x, int ld_x, int Tin, int dt, float* y, int ld_y, int Tout, int stride,
              int padding, int dilation, const float* res, int ld_res, int res_shift, float scale, int accumulate,
              int out_row_shift = 0, int mirror = 0, int epi_gelu = 0) {
        if (!live()) return;
        ConvArgs a;
        if (!fill_args(a, w, Tin, Tout, stride, padding, dilation, out_row_shift)) return;
        a.res = res; a.ld_res = ld_res; a.res_shift = res_shift;
        a.y = y; a.ld_y = ld_y;
        a.scale = scale; a.accumulate = accumulate; a.mirror = mirror;
        a.epi_gelu = epi_gelu;                   // tensor-core path only: y is the 16-bit GELU output (the caller checked use_tc)
        if (epi_gelu && !use_tc(w, dt) && err == ST2_OK) {
            set_error("conv: the GELU epilogue exists on the tensor-core path only");
            err = ST2_ERR_STATE;
            return;
        }
        // a pointwise conv (k = 1: the Linear layers, LSTM input projections, shortcuts) has no halo: the B utterances are one
        // dense [B*T] row range, so no 128-row tile is left partly empty at the end of every utterance (T = 400: 22 % of the tiles)
        if (w.k == 1 && !w.transposed && stride == 1 && padding == 0 && out_row_shift == 0 && res_shift == 0 && !mirror &&
            Tin == Tout && (int64_t)B * Tout < (int64_t)1 << 30) {
            a.B = 1;
            a.Tin = a.Tout = a.M = B * Tout;
        }
        // algorithmic work (SURVEY.md 8(d)): Conv1d 2*B*Tout*Cout*Cin*k ; ConvTranspose1d 2*B*Tin*Cin*Cout*k
        const double flops = 2.0 * B * (w.transposed ? (double)Tin : (double)(Tout - out_row_shift)) * w.Cin * w.Cout * w.k;
        const bool tc = use_tc(w, dt);
        const double bytes = (double)B * ((double)w.Cin * Tin * (tc ? 2 : 4) +
                                          (double)w.Cout * Tout * (epi_gelu ? 2 : 4) * (1 + (res ? 1 : 0) + (accumulate ? 1 : 0))) +
                             (double)w.k * w.Cin * w.Cout * (tc ? 2 : 4);
        if (tc) {
            a.x16 = x; a.ld_x16 = ld_x; a.w16 = w.w16[dt]; a.w16_cin_pad = w.cin_pad; a.w16_cout_pad = w.cout_pad;
            a.fmt16 = dt;
            chk(launch_conv_tc(a, st));
            prof(PC_CONV_TC, flops, bytes);
        } else {
            a.x = (const float*)x; a.ld_x = ld_x;
            chk(launch_conv_simt(a, st));
            prof(PC_CONV_SIMT, flops, bytes);
        }
    }

    // ---- fused path: statistics references, coefficient kernels, fused conv ---------------------
    // f2: float2 tile partials (conv_pipe / conv_fused epilogues); row: per-(CTA, utterance, warp) partials of conv_row.cu,
    // located by `rd`; neither: double2 slab partials of the standalone statistics pass
    // shift: the partials are of x - shift[c] (float2 tile partials only)
    struct StatRef { const void* ptr; int nparts; bool f2; bool row = false; RowStatsDesc rd = {}; const float* shift = nullptr; };
    bool last_row = false;        // did the last conv_fused() run on conv_row.cu (statistics in its layout)?
    RowStatsDesc last_rd = {};
    StatRef produced(const void* buf, int nparts) const {
        StatRef r{buf, nparts, true};
        r.row = last_row;
        r.rd = last_rd;
        return r;
    }

    // statistics of a tensor no fused epilogue produced (noise_convs output): standalone pass
    StatRef stats_standalone(const float* x, int ld_x, int T, int C) {
        void* scratch = alloc(adain_scratch_bytes(B, T, C));
        if (live()) {
            chk(launch_in_stats(x, ld_x, B, T, C, scratch, st));
            prof(PC_NORM_STATS, 0, (double)B * T * C * 4);
        }
        return StatRef{scratch, 0, false};
    }
    // coef <- (1+gamma)*rstd, beta - mean*(1+gamma)*rstd  (n == nullptr: identity)
    static constexpr int kCoefMax = 2048;     // channels per utterance the coefficient buffer holds (allocated as B*2*2048)
    // x_offset: the tensor is stored as x - x_offset[c] (the bias-free fp16 noise source); only for float2 tile partials
    void coef_from(const StatRef& sr, const AdaINRef* n, int T, int C, int Cpad, const float* x_offset = nullptr) {
        if (!live()) return;
        if ((x_offset != nullptr || sr.shift != nullptr) && (n == nullptr || !sr.f2 || sr.row)) {
            set_error("coef_from: an input offset or statistics shift needs float2 tile partials");
            err = ST2_ERR_STATE;
            return;
        }
        if (Cpad > kCoefMax) {
            set_error("coefficient buffer holds %d channels, layer needs %d", kCoefMax, Cpad);
            err = ST2_ERR_UNSUPPORTED;
            return;
        }
        if (n == nullptr || !sr.f2)
            chk(launch_adain_coef(n ? sr.ptr : nullptr, n ? H : nullptr, d->fc_rows, n ? n->h_off : 0, coef, B, T, C, Cpad, st));
        else if (sr.row)
            chk(launch_adain_coef_row(sr.ptr, sr.rd, H, d->fc_rows, n->h_off, coef, B, T, C, Cpad, st));
        else
            chk(launch_adain_coef_f2(sr.ptr, sr.nparts, H, d->fc_rows, n->h_off, coef, B, T, C, Cpad, st, x_offset, sr.shift));
        prof(PC_NORM_COEF, 0, 0);
        coef_ld = Cpad;
    }
    bool can_fuse(const ConvW& w, int dt, int ld_x, int ld_y, int stride, int dilation) {
        if (!use_tc(w, dt)) return false;
        ConvArgs a;
        memset(&a, 0, sizeof(a));
        a.in_stride = 1; a.w16 = w.w16[dt]; a.w16_cin_pad = w.cin_pad; a.w16_cout_pad = w.cout_pad;
        a.Cin = w.Cin; a.Cout = w.Cout; a.ld_x = ld_x; a.ld_y = ld_y; a.ld_res = 4;
        a.ntaps = w.transposed ? w.k / stride : w.k;
        a.tap_step = w.transposed ? -1 : dilation;
        return conv_fused_supported(a);
    }
    // a fused conv's ConvArgs but for its buffers (x, y, res, acc_src), which the launch fills in: geometry, 16-bit weights,
    // residual pitch ld_y, epilogue scale 1; shift: the output is written one row down and row 2 mirrored into row 0
    ConvArgs fused_args(const ConvW& w, int dt, int ld_x, int Tin, int ld_y, int Tout, int stride, int padding, int dilation,
                        int shift = 0) {
        ConvArgs a;
        fill_args(a, w, Tin, Tout, stride, padding, dilation, shift);
        a.ld_x = ld_x; a.ld_y = ld_y; a.ld_res = ld_y;
        a.scale = 1.f; a.mirror = shift;
        a.w16 = w.w16[dt]; a.w16_cin_pad = w.cin_pad; a.w16_cout_pad = w.cout_pad; a.fmt16 = dt;
        return a;
    }
    // would a planned launch run on conv_pipe.cu?  ConvArgs tells a residual (res) and a separate source of the old values
    // (acc16) by non-null pointers, and a plan is made before its buffers exist (and in the workspace dry run, which has none),
    // so they are marked with kPlanned here
    static constexpr float kPlanned = 0.f;
    bool on_pipe(ConvArgs a, bool res) {
        if (res) a.res = &kPlanned;
        if (a.acc16) a.acc_src = &kPlanned;
        return conv_pipe_supported(a);
    }
    // AdaIN of a fused conv's input: the statistics of the input, the AdaIN, and `off` when the input is stored as x - off[c]
    struct AdaIn { StatRef sr; const AdaINRef* n; const float* off = nullptr; };
    // y = epilogue( conv( act(coef.a * x + coef.b) ) ), statistics of y -> stats_out (float2 partials)
    void conv_fused(const ConvArgs& a, int act, float slope, const float* alpha, void* stats_out, const AdaIn* in = nullptr) {
        // with `in`, the coefficients of the input transform come from it: when both the producer of the statistics and this conv
        // run on conv_row.cu the kernel computes them itself (no launch in between); otherwise the coefficient kernel is launched
        // here, as coef_from() before the call would
        if (!live()) return;
        // the kernel, decided once: the 32 / 64-channel Snake convs on fp16 tensors run on the row-per-thread kernel (conv_row.cu;
        // its statistics partials have their own layout, recorded in last_rd for the coefficient kernel), the rest on conv_pipe.cu
        // where it takes them, else on conv_fused.cu
        const int cat = (act == ACT_SNAKE && conv_row_supported(a)) ? PC_CONV_ROW : conv_pipe_supported(a) ? PC_CONV_PIPE : PC_CONV_FUSED;
        const bool row = cat == PC_CONV_ROW;
        RowCoefSrc src{};
        bool inline_coef = false;
        if (in != nullptr) {
            inline_coef = row && in->n != nullptr && in->sr.f2 && in->sr.row && in->off == nullptr && conv_row_inline_coef_ok(a);
            if (inline_coef) src = RowCoefSrc{in->sr.ptr, in->sr.rd, H, d->fc_rows, in->n->h_off, a.Tin};
            else coef_from(in->sr, in->n, a.Tin, a.Cin, a.Cin, in->off);
            if (err != ST2_OK) return;
        }
        last_row = row;
        if (row) chk(launch_conv_row(a, coef, coef_ld, act, alpha, stats_out, &last_rd, st, inline_coef ? &src : nullptr));
        else if (cat == PC_CONV_PIPE) chk(launch_conv_pipe(a, coef, coef_ld, act, slope, alpha, stats_out, st));
        else chk(launch_conv_fused(a, coef, coef_ld, act, slope, alpha, stats_out, st));
        // algorithmic work as in conv(): k = w_step * ntaps taps; a transposed conv (tap_step -1) counts its Tin input rows
        const int k = a.w_step * a.ntaps;
        const double flops = 2.0 * B * (a.tap_step < 0 ? (double)a.Tin : (double)a.Tout) * a.Cin * a.Cout * k;
        const double bytes = (double)B * ((double)a.Cin * a.Tin * (a.x16in ? 2 : 4) +
                                          (double)a.Cout * a.Tout * ((a.y16out ? 2 : 4) + (a.res ? (a.res16 ? 2 : 4) : 0) +
                                                                     (a.accumulate ? (a.acc16 ? 2 : 4) : 0))) +
                             (double)k * a.Cin * a.Cout * 2;
        prof(cat, flops, bytes);
    }

    // AdainResBlk1d.forward (hifigan.py:400-403).  x [B,T,ld_x] (Cin real channels) -> y [B,T or 2T,ld_y]
    void resblk1d(const ResBlk1dW& w, const float* x, int ld_x, int T, float* y, int ld_y) {
        const int64_t mark = off;
        const int dt = fmt_for(w.name);
        const bool tc1 = use_tc(w.conv1, dt);
        const int dt1 = tc1 ? dt : DT_F32;
        const int dta = (tc1 && !w.upsample) ? dt : DT_F32;     // the depthwise pool reads fp32, writes the 16-bit operand
        const int es1 = dta == DT_F32 ? 4 : 2;
        const int Tc = w.upsample ? 2 * T : T;
        void* xa = alloc((int64_t)B * T * ld_x * es1);
        norm_act(x, ld_x, T, w.Cin, &w.norm1, ACT_LRELU, 0.2f, nullptr, xa, ld_x, dta);
        const void* cin = xa;
        if (w.upsample) {
            void* xp = alloc((int64_t)B * Tc * ld_x * (tc1 ? 2 : 4));
            if (live()) {
                if (tc1) chk(launch_pool_dw16((const float*)xa, ld_x, w.pool_w, w.pool_b, xp, ld_x, dt, B, T, ld_x, st));
                else chk(launch_pool_dw((const float*)xa, ld_x, w.pool_w, w.pool_b, (float*)xp, ld_x, B, T, w.Cin, ld_x, st));
            }
            prof(PC_MISC, 0, 4.0 * B * w.Cin * 3.0 * T);
            cin = xp;
        }
        float* h1 = allocf((int64_t)B * Tc * w.Cout);
        conv(w.conv1, cin, ld_x, Tc, dt1, h1, w.Cout, Tc, 1, 1, 1, nullptr, 0, 0, 1.f, 0);
        tap(w.name + ".conv1", h1, w.Cout, (int64_t)B * Tc, w.Cout);
        const bool tc2 = use_tc(w.conv2, dt);
        const int dt2 = tc2 ? dt : DT_F32;
        void* xa2 = alloc((int64_t)B * Tc * w.Cout * (dt2 == DT_F32 ? 4 : 2));
        norm_act(h1, w.Cout, Tc, w.Cout, &w.norm2, ACT_LRELU, 0.2f, nullptr, xa2, w.Cout, dt2);
        const float* res = x;
        int ld_res = ld_x;
        if (w.has_sc) {
            float* sc = allocf((int64_t)B * T * w.Cout);
            const bool tcs = use_tc(w.conv1x1, dt);
            const void* xin = x;
            if (tcs) {   // 16-bit copy of the raw block input for the tensor-core 1x1
                void* x16 = alloc((int64_t)B * T * ld_x * 2);
                norm_act(x, ld_x, T, w.Cin, nullptr, ACT_NONE, 0.f, nullptr, x16, ld_x, dt);
                xin = x16;
            }
            conv(w.conv1x1, xin, ld_x, T, tcs ? dt : DT_F32, sc, w.Cout, T, 1, 0, 1, nullptr, 0, 0, 1.f, 0);
            res = sc;
            ld_res = w.Cout;
        }
        conv(w.conv2, xa2, w.Cout, Tc, dt2, y, ld_y, Tc, 1, 1, 1, res, ld_res, w.upsample ? 1 : 0,
             0.70710678118654752f, 0);
        tap(w.name, y, ld_y, (int64_t)B * Tc, w.Cout);
        off = mark;
    }

    // ---- fp16 storage of a generator stage ---------------------------------------------------------------------------
    // how a fused AdaINResBlock1 runs (plan_stage): its part in the stage's sum and which of its tensors are stored as fp16
    struct BlockPlan {
        bool fused = false;      // on the fused conv kernels; else the coefficient / affine kernels and conv()
        int accumulate = 0;      // the last conv adds the old values of dest ...
        float scale = 1.f;       // ... and scales the sum (the last block of a stage: the mean over the blocks)
        bool xt16 = false;       // the intra-block tensor xt
        bool run16 = false;      // the running tensor between the iterations (needs xt16)
        bool x16 = false;        // the block input (needs run16)
        int sum16 = 0;           // the stage's partial sum, of which the block is the 1 first, 2 middle or 3 last (needs run16)
        bool dest16 = false;     // dest (needs sum16 == 3)
    };
    struct StagePlan {
        ConvArgs ups;            // generator.ups[i] on the fused path, but for its buffers
        bool ups_fused = false;
        BlockPlan src;           // generator.noise_res[i]
        BlockPlan res[3];        // generator.resblocks[i * 3 + j] (n_kernels is 3, st2_decoder_create)
    };
    // convs1[j] (c2 = false) or convs2[j] of fused block w run with plan p, but for its buffers: x, y, the running tensor
    // (residual of convs2) and, with acc16, the stage's fp16 sum (old values of the last convs2)
    ConvArgs block_args(const ResBlock1W& w, const BlockPlan& p, int j, bool c2, int T) {
        const int dil = c2 ? 1 : w.dil[j], run16 = j > 0 ? p.run16 : p.x16;    // the running tensor: the block input at j = 0
        ConvArgs a = fused_args(c2 ? w.c2[j] : w.c1[j], fmt_for(w.name), w.C, T, w.C, T, 1, (w.k * dil - dil) / 2, dil);
        a.x16in = c2 ? p.xt16 : run16;
        a.y16out = !c2 ? p.xt16 : j < 2 ? p.run16 : (p.sum16 != 0 && (p.sum16 < 3 || p.dest16));
        a.res16 = c2 ? run16 : 0;
        if (c2 && j == 2) { a.accumulate = p.accumulate; a.scale = p.scale; a.acc16 = p.sum16 > 1 ? 1 : 0; }
        return a;
    }
    bool block_on_pipe(const ResBlock1W& w, const BlockPlan& p, int T) {
        for (int j = 0; j < 3; ++j)
            if (!on_pipe(block_args(w, p, j, false, T), false) || !on_pipe(block_args(w, p, j, true, T), true)) return false;
        return true;
    }
    // The fp16 storage of generator stage i at T rows (DESIGN.md section 3), the only reader of the options fp16_storage and
    // fp16_*.  A tensor private to the stage is stored as fp16 when every conv that touches it still runs on conv_pipe.cu with
    // it; its AdaIN statistics still come from the fp32 values in the producing epilogue.  ups: the fused ups conv but for its
    // buffers and y16out.
    StagePlan plan_stage(int i, int T, const ConvArgs& ups) {
        const st2_config& c = d->cfg;
        const int n = c.n_kernels;
        const bool istft = c.variant == 1;
        const ResBlock1W& nr = d->noise_res[i];
        const ResBlock1W* rb = &d->resblocks[i * n];
        // (1) xt, conv1's output, read only by conv2's transform: 20 % fewer HBM bytes per iteration for -0.1 dB of SNR
        // (fp16_xt = 0 turns off every kind)
        auto block = [&](const ResBlock1W& w, int accumulate, float scale) {
            BlockPlan p;
            p.fused = can_fuse(w.c1[0], fmt_for(w.name), w.C, w.C, 1, 5);
            p.accumulate = accumulate; p.scale = scale;
            p.xt16 = p.fused && d->fp16_storage && d->opt_xt16;
            p.xt16 = p.xt16 && block_on_pipe(w, p, T);
            return p;
        };
        // (2) the running tensor between the three iterations (x + conv2 output of iterations 0 and 1, read as the next conv1's
        // input and conv2's residual; the block output stays fp32): 25 % fewer bytes per block (fp16_run); x16: with an fp16
        // block input, which needs the statistics of its producer
        auto takes16 = [&](const ResBlock1W& w, BlockPlan p, bool x16) {
            p.run16 = p.xt16 && d->opt_run16;
            p.x16 = p.run16 && x16;
            return p.run16 && block_on_pipe(w, p, T);
        };
        auto input16 = [&](const ResBlock1W& w, BlockPlan& p, bool x16) { p.x16 = x16; p.run16 = x16 || takes16(w, p, false); };
        StagePlan sp;
        // (5) the noise_convs output, input of noise_res (conv1 input and residual of its first iteration), stored without its
        // bias; the istftnet source conv writes no statistics (fp16_src)
        sp.src = block(nr, 0, 1.f);
        input16(nr, sp.src, !istft && d->opt_src16 && takes16(nr, sp.src, true));
        // (3) the stage input xu = ups(x) + x_source, read six times (input and residual of the first iteration of the three
        // blocks), written by the ups conv (fp16_xu)
        sp.ups = ups;
        sp.ups.y16out = 1;
        sp.ups_fused = can_fuse(d->ups[i], ups.fmt16, ups.ld_x, ups.ld_y, c.upsample_rates[i], 1);
        bool xu16 = sp.ups_fused && d->opt_xu16 && on_pipe(sp.ups, true);
        for (int j = 0; j < n; ++j) sp.res[j] = block(rb[j], j > 0 ? 1 : 0, j + 1 == n ? 1.f / (float)n : 1.f);
        for (int j = 0; j < n; ++j) xu16 = xu16 && takes16(rb[j], sp.res[j], true);
        sp.ups.y16out = xu16 ? 1 : 0;
        for (int j = 0; j < n; ++j) input16(rb[j], sp.res[j], xu16);
        // (4) the partial sum over the blocks, written by the first, read and written in place by the middle ones, read by the
        // last, which writes the stage output: these accumulate layers sit at their byte floor (fp16_sum)
        bool sum16 = n >= 2 && d->opt_sum16;
        for (int j = 0; j < n; ++j) sp.res[j].sum16 = j == 0 ? 1 : (j + 1 == n ? 3 : 2);
        for (int j = 0; j < n && sum16; ++j) sum16 = sp.res[j].run16 && block_on_pipe(rb[j], sp.res[j], T);
        for (int j = 0; j < n && !sum16; ++j) sp.res[j].sum16 = 0;
        // (6) the last stage's output, read only by conv_post's kernel (fp16_out)
        BlockPlan& lb = sp.res[n - 1];
        lb.dest16 = sum16 && i + 1 == c.n_stages && !istft && d->opt_out16;
        lb.dest16 = lb.dest16 && block_on_pipe(rb[n - 1], lb, T);
        return sp;
    }

    // AdaINResBlock1.forward (hifigan.py:65-74) on x_in [B,T,C] run with plan p; the running tensor lives in `run` (may alias
    // x_in for an in-place block); the last iteration writes dest = (dest_old*accumulate + conv2 + run) * scale, through the
    // stage's fp16 partial sum sum16buf when p.sum16.  in_stats: statistics of x_in from its producer (else a standalone pass).
    // x_offset / c2b0: x_in is stored as x - x_offset[c]; c2b0 = c2[0].bias + x_offset puts it back in the residual add
    void resblock1(const ResBlock1W& w, const BlockPlan& p, const float* x_in, float* run, int T, float* dest,
                   const StatRef* in_stats = nullptr, void* sum16buf = nullptr, const float* x_offset = nullptr,
                   const float* c2b0 = nullptr) {
        const int64_t mark = off;
        const int C = w.C;
        const int dt = fmt_for(w.name);
        if (p.fused) {
            // fused: 2 tiny coefficient kernels + 2 fused convs per iteration; AdaIN statistics come from the
            // producing conv's epilogue (or from in_stats for the block input)
            const int nparts = fused_stats_parts(block_args(w, p, 0, false, T));
            int64_t st_bytes = (int64_t)B * nparts * C * 8;
            if ((C == 32 || C == 64) && conv_row_stats_bytes(B, T, C) > st_bytes) st_bytes = conv_row_stats_bytes(B, T, C);
            void* st_xt = alloc(st_bytes);
            void* st_run = alloc(st_bytes);
            float* xt = (float*)alloc((int64_t)B * T * C * 4);      // sized for fp32 (the dry run must not depend on the device)
            void* r16buf = alloc((int64_t)B * T * C * 2);           // allocated either way: same workspace on every device
            StatRef cur_st = in_stats ? *in_stats : stats_standalone(x_in, C, T, C);
            const float* cur = x_in;
            for (int j = 0; j < 3; ++j) {
                const bool last = (j == 2);
                ConvArgs a1 = block_args(w, p, j, false, T);
                a1.x = cur; a1.y = xt;
                const AdaIn in1{cur_st, &w.n1[j], j == 0 ? x_offset : nullptr};
                conv_fused(a1, ACT_SNAKE, 0.f, w.alpha1[j], st_xt, &in1);
                if (!p.xt16) tap(w.name + ".convs1." + std::to_string(j), xt, C, (int64_t)B * T, C);
                else tap16(w.name + ".convs1." + std::to_string(j), xt, (int64_t)B * T * C);
                ConvArgs a2 = block_args(w, p, j, true, T);
                float* out = last ? ((p.sum16 == 1 || p.sum16 == 2) ? (float*)sum16buf : dest) : (p.run16 ? (float*)r16buf : run);
                a2.x = xt; a2.y = out; a2.res = cur;
                if (a2.acc16) a2.acc_src = sum16buf;
                if (j == 0 && x_offset != nullptr) a2.bias = c2b0;
                const AdaIn in2{produced(st_xt, nparts), &w.n2[j]};
                conv_fused(a2, ACT_SNAKE, 0.f, w.alpha2[j], last ? nullptr : st_run, &in2);
                if (a2.y16out && !(last && p.dest16)) tap16(w.name + ".iter" + std::to_string(j), out, (int64_t)B * T * C);
                else if (!last || (!p.accumulate && p.scale == 1.f)) tap(w.name + ".iter" + std::to_string(j), out, C, (int64_t)B * T, C);
                cur = out;
                cur_st = produced(st_run, nparts);
            }
            off = mark;
            return;
        }
        const bool tc = use_tc(w.c1[0], dt);
        const int dta = tc ? dt : DT_F32;
        void* xa = alloc((int64_t)B * T * C * (dta == DT_F32 ? 4 : 2));
        float* xt = allocf((int64_t)B * T * C);
        const float* cur = x_in;
        for (int j = 0; j < 3; ++j) {
            const int dil = w.dil[j];
            norm_act(cur, C, T, C, &w.n1[j], ACT_SNAKE, 0.f, w.alpha1[j], xa, C, dta);
            conv(w.c1[j], xa, C, T, dta, xt, C, T, 1, (w.k * dil - dil) / 2, dil, nullptr, 0, 0, 1.f, 0);
            tap(w.name + ".convs1." + std::to_string(j), xt, C, (int64_t)B * T, C);
            norm_act(xt, C, T, C, &w.n2[j], ACT_SNAKE, 0.f, w.alpha2[j], xa, C, dta);
            const bool last = (j == 2);
            float* out = last ? dest : run;
            conv(w.c2[j], xa, C, T, dta, out, C, T, 1, (w.k - 1) / 2, 1, cur, C, 0, last ? p.scale : 1.f,
                 last ? p.accumulate : 0);
            if (!last || (!p.accumulate && p.scale == 1.f)) tap(w.name + ".iter" + std::to_string(j), out, C, (int64_t)B * T, C);
            cur = out;
        }
        off = mark;
    }
};

}  // namespace st2
