"""Helpers for the -m gpu tests: thin ctypes callers of the unit entry points + diagnostics log."""
import ctypes as C
import json
import os

import numpy as np
import torch

from styletts2_lite_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "gpurun_out")


def log(name, **kv):
    """Append one JSON line of parity metrics to gpurun_out/parity.jsonl (read back by the author)."""
    try:
        os.makedirs(OUT, exist_ok=True)
        with open(os.path.join(OUT, "parity.jsonl"), "a") as f:
            f.write(json.dumps(dict(test=name, **{k: (float(v) if isinstance(v, (np.floating, float)) else v)
                                                  for k, v in kv.items()})) + "\n")
    except OSError:
        pass


def dev():
    return torch.device("cuda", 0)


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def to_dev(a, dtype=torch.float32):
    return torch.from_numpy(np.ascontiguousarray(a)).to(device=dev(), dtype=dtype).contiguous()


def cl(x_bct):
    """[B,C,T] numpy -> channels-last contiguous [B,T,C]."""
    return np.ascontiguousarray(np.transpose(x_bct, (0, 2, 1)))


def cf(x_btc):
    return np.ascontiguousarray(np.transpose(x_btc, (0, 2, 1)))


def sinegen_phase(f0, scale):
    lib = _lib.load()
    B, L2 = f0.shape
    f0d = to_dev(f0)
    phase = torch.empty(B, L2 * scale, 9, device=dev())
    frames = torch.empty(B, L2, 9, device=dev())
    _lib.check(lib.st2_sinegen_phase(_lib.ptr(f0d), _lib.ptr(phase), _lib.ptr(frames), B, L2, scale, stream()), "sinegen_phase")
    torch.cuda.synchronize()
    return phase.cpu().numpy(), frames.cpu().numpy()


def har_source(f0, noise, lin_w, lin_b, scale, seed=0):
    lib = _lib.load()
    B, L2 = f0.shape
    f0d = to_dev(f0)
    nz = None if noise is None else to_dev(noise)
    w, b = to_dev(lin_w.reshape(-1)), to_dev(lin_b.reshape(-1))
    har = torch.empty(B, L2 * scale, device=dev())
    frames = torch.empty(B, L2, 9, device=dev())
    _lib.check(lib.st2_har_source(_lib.ptr(f0d), _lib.ptr(nz), C.c_uint64(seed), _lib.ptr(w), _lib.ptr(b), _lib.ptr(har),
                                  _lib.ptr(frames), B, L2, scale, stream()), "har_source")
    torch.cuda.synchronize()
    return har.cpu().numpy()


def adain_act(x_btc, h, alpha, act, slope=0.0, out_dtype="fp32", ld_pad=0):
    """x channels-last [B,T,C]; h [B,2C] or None; returns fp32 numpy [B,T,C]."""
    lib = _lib.load()
    B, T, Cc = x_btc.shape
    ld = Cc + ld_pad
    xd = torch.zeros(B, T, ld, device=dev())
    xd[:, :, :Cc] = to_dev(x_btc)
    hd = None if h is None else to_dev(h)
    ad = None if alpha is None else to_dev(alpha.reshape(-1))
    tdt = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}[out_dtype]
    y = torch.zeros(B, T, ld, device=dev(), dtype=tdt)
    nbytes = _lib.check(lib.st2_adain_scratch_bytes(B, T, Cc), "adain_scratch_bytes")
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev())
    _lib.check(lib.st2_adain_act(_lib.ptr(xd), ld, _lib.ptr(hd), 0 if h is None else h.shape[1], _lib.ptr(ad),
                                 _lib.ACT[act], C.c_float(slope), _lib.ptr(y), ld, _lib.DTYPE[out_dtype], B, T, Cc,
                                 _lib.ptr(scratch), stream()), "adain_act")
    torch.cuda.synchronize()
    return y[:, :, :Cc].float().cpu().numpy()


def conv1d(x_btc, w, bias, stride=1, padding=0, dilation=1, output_padding=0, transposed=False, precision="fp32"):
    """x channels-last [B,T,Cin]; w in the reference layout; returns channels-last [B,Tout,Cout]."""
    lib = _lib.load()
    B, T, Cin = x_btc.shape
    k = w.shape[2]
    Cout = w.shape[1] if transposed else w.shape[0]
    if transposed:
        Tout = (T - 1) * stride - 2 * padding + (k - 1) + output_padding + 1
    else:
        Tout = (T + 2 * padding - dilation * (k - 1) - 1) // stride + 1
    xd, wd = to_dev(x_btc), to_dev(w)
    bd = None if bias is None else to_dev(bias)
    y = torch.full((B, Tout, Cout), float("nan"), device=dev())
    prec = _lib.PREC[precision]
    nbytes = _lib.check(lib.st2_conv1d_scratch_bytes(B, T, Cin, Cout, k, prec), "conv1d_scratch_bytes")
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev())
    _lib.check(lib.st2_conv1d(_lib.ptr(xd), _lib.ptr(wd), _lib.ptr(bd), _lib.ptr(y), _lib.ptr(scratch), B, T, Cin, Cout, k,
                              stride, padding, dilation, output_padding, 1 if transposed else 0, prec, stream()), "conv1d")
    torch.cuda.synchronize()
    return y.cpu().numpy()


def adain_conv1d_fused(x_btc, h, alpha, act, w, bias, res_btc, y_old_btc, h_next, padding, dilation, scale=1.0,
                       slope=0.0, precision="bf16"):
    """Fused half-step of AdaINResBlock1 on channels-last tensors; returns (y [B,T,Cout], coef_next [B,2,Cout] or None)."""
    lib = _lib.load()
    B, T, Cin = x_btc.shape
    Cout, _, k = w.shape
    xd, wd = to_dev(x_btc), to_dev(w)
    hd = None if h is None else to_dev(h)
    ad = None if alpha is None else to_dev(alpha.reshape(-1))
    bd = None if bias is None else to_dev(bias)
    rd = None if res_btc is None else to_dev(res_btc)
    hn = None if h_next is None else to_dev(h_next)
    cn = None if h_next is None else torch.full((B, 2, Cout), float("nan"), device=dev())
    if y_old_btc is None:
        y = torch.full((B, T, Cout), float("nan"), device=dev())
    else:
        y = to_dev(y_old_btc)
    nbytes = _lib.check(lib.st2_adain_conv1d_fused_scratch_bytes(B, T, Cin, Cout, k), "fused_scratch_bytes")
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev())
    _lib.check(lib.st2_adain_conv1d_fused(_lib.ptr(xd), _lib.ptr(hd), _lib.ptr(ad), _lib.ACT[act], C.c_float(slope),
                                          _lib.ptr(wd), _lib.ptr(bd), _lib.ptr(rd), _lib.ptr(y), _lib.ptr(hn), _lib.ptr(cn),
                                          _lib.ptr(scratch), B, T, Cin, Cout, k, padding, dilation, C.c_float(scale),
                                          0 if y_old_btc is None else 1, _lib.PREC[precision], stream()),
               "adain_conv1d_fused")
    torch.cuda.synchronize()
    return y.cpu().numpy(), (None if cn is None else cn.cpu().numpy())


def adain_conv1d_row(x_btc, h, alpha, w, bias, res_btc, old_btc, h_next, padding, dilation, scale=1.0, precision="bf16",
                     x16=True, y16=True):
    """The same half-step on conv_row.cu (fp16 residual / old values added by the tensor core); returns (y, coef_next)."""
    lib = _lib.load()
    B, T, Cc = x_btc.shape
    k = w.shape[2]
    xd, wd, hd, ad = to_dev(x_btc), to_dev(w), to_dev(h), to_dev(alpha.reshape(-1))
    bd = None if bias is None else to_dev(bias)
    rd = None if res_btc is None else to_dev(res_btc)
    od = None if old_btc is None else to_dev(old_btc)
    hn = None if h_next is None else to_dev(h_next)
    cn = None if h_next is None else torch.full((B, 2, Cc), float("nan"), device=dev())
    y = torch.full((B, T, Cc), float("nan"), device=dev())
    nbytes = _lib.check(lib.st2_adain_conv1d_row_scratch_bytes(B, T, Cc, k), "row_scratch_bytes")
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev())
    _lib.check(lib.st2_adain_conv1d_row(_lib.ptr(xd), _lib.ptr(hd), _lib.ptr(ad), _lib.ptr(wd), _lib.ptr(bd), _lib.ptr(rd),
                                        _lib.ptr(od), _lib.ptr(y), _lib.ptr(hn), _lib.ptr(cn), _lib.ptr(scratch), B, T, Cc, k,
                                        padding, dilation, C.c_float(scale), _lib.PREC[precision], 1 if x16 else 0,
                                        1 if y16 else 0, stream()), "adain_conv1d_row")
    torch.cuda.synchronize()
    return y.cpu().numpy(), (None if cn is None else cn.cpu().numpy())


def adain_conv1d_row_pair(x_btc, h1, alpha1, w1, b1, h2, alpha2, w2, b2, h_next, dil1, dil2, precision="bf16"):
    """Two chained half-steps on conv_row.cu (y1 = step(x), y2 = step(y1) + x, x stored as fp16); returns
    (y1, y2, coef_next, inline) with y1 / y2 channels-last [B,T,C] and `inline` whether the second launch computed the AdaIN
    coefficients of y1 itself."""
    lib = _lib.load()
    B, T, Cc = x_btc.shape
    k1, k2 = w1.shape[2], w2.shape[2]
    xd, h1d, a1d, w1d = to_dev(x_btc), to_dev(h1), to_dev(alpha1.reshape(-1)), to_dev(w1)
    h2d, a2d, w2d = to_dev(h2), to_dev(alpha2.reshape(-1)), to_dev(w2)
    b1d = None if b1 is None else to_dev(b1)
    b2d = None if b2 is None else to_dev(b2)
    hn = None if h_next is None else to_dev(h_next)
    cn = None if h_next is None else torch.full((B, 2, Cc), float("nan"), device=dev())
    y1 = torch.full((B, T, Cc), float("nan"), device=dev())
    y2 = torch.full((B, T, Cc), float("nan"), device=dev())
    inline = C.c_int32(-1)
    nbytes = _lib.check(lib.st2_adain_conv1d_row_pair_scratch_bytes(B, T, Cc, k1, k2), "row_pair_scratch_bytes")
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev())
    _lib.check(lib.st2_adain_conv1d_row_pair(_lib.ptr(xd), _lib.ptr(h1d), _lib.ptr(a1d), _lib.ptr(w1d), _lib.ptr(b1d),
                                             _lib.ptr(h2d), _lib.ptr(a2d), _lib.ptr(w2d), _lib.ptr(b2d), _lib.ptr(y1), _lib.ptr(y2),
                                             _lib.ptr(hn), _lib.ptr(cn), C.byref(inline), _lib.ptr(scratch), B, T, Cc, k1, dil1,
                                             k2, dil2, _lib.PREC[precision], stream()), "adain_conv1d_row_pair")
    torch.cuda.synchronize()
    return y1.cpu().numpy(), y2.cpu().numpy(), (None if cn is None else cn.cpu().numpy()), inline.value == 1


def act_conv_transpose1d_fused(x_btc, alpha, act, w, bias, res_btc, h_next, stride, padding, output_padding, slope=0.0,
                               precision="bf16"):
    """Fused upsampling step on channels-last tensors; returns (y [B,Tout,Cout], coef_next [B,2,Cout] or None)."""
    lib = _lib.load()
    B, T, Cin = x_btc.shape
    _, Cout, k = w.shape
    Tout = (T - 1) * stride - 2 * padding + (k - 1) + output_padding + 1
    xd, wd = to_dev(x_btc), to_dev(w)
    ad = None if alpha is None else to_dev(alpha.reshape(-1))
    bd = None if bias is None else to_dev(bias)
    rd = None if res_btc is None else to_dev(res_btc)
    hn = None if h_next is None else to_dev(h_next)
    cn = None if h_next is None else torch.full((B, 2, Cout), float("nan"), device=dev())
    y = torch.full((B, Tout, Cout), float("nan"), device=dev())
    nbytes = _lib.check(lib.st2_act_conv_transpose1d_fused_scratch_bytes(B, T, Cin, Cout, k, stride), "fused_t_scratch_bytes")
    # the residual view of the kernel may read (never use) a few rows before / after the tensor: keep it inside one arena
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev())
    _lib.check(lib.st2_act_conv_transpose1d_fused(_lib.ptr(xd), _lib.ptr(ad), _lib.ACT[act], C.c_float(slope), _lib.ptr(wd),
                                                  _lib.ptr(bd), _lib.ptr(rd), _lib.ptr(y), _lib.ptr(hn), _lib.ptr(cn),
                                                  _lib.ptr(scratch), B, T, Cin, Cout, k, stride, padding, output_padding,
                                                  _lib.PREC[precision], stream()), "act_conv_transpose1d_fused")
    torch.cuda.synchronize()
    return y.cpu().numpy(), (None if cn is None else cn.cpu().numpy())


def adain_conv1d_fused_ex(x_btc, h, alpha, act, w, bias, res_btc, old_btc, y_old_btc, h_next, padding, dilation, scale=1.0,
                          slope=0.0, precision="bf16", x16=False, res16=False, old16=False, y16=False, old_in_y=False):
    """st2_adain_conv1d_fused_ex: the fused half-step with the decoder's fp16 storage types.  old_btc is the separate accumulate
    source (stored as fp16 when old16; with old_in_y it is first stored into the fp16 y and the conv accumulates in place);
    y_old_btc the old values of y for the plain accumulate.  Returns (y [B,T,Cout], coef_next [B,2,Cout] or None)."""
    lib = _lib.load()
    B, T, Cin = x_btc.shape
    Cout, _, k = w.shape
    xd, wd = to_dev(x_btc), to_dev(w)
    hd = None if h is None else to_dev(h)
    ad = None if alpha is None else to_dev(alpha.reshape(-1))
    bd = None if bias is None else to_dev(bias)
    rd = None if res_btc is None else to_dev(res_btc)
    od = None if old_btc is None else to_dev(old_btc)
    hn = None if h_next is None else to_dev(h_next)
    cn = None if h_next is None else torch.full((B, 2, Cout), float("nan"), device=dev())
    y = torch.full((B, T, Cout), float("nan"), device=dev()) if y_old_btc is None else to_dev(y_old_btc)
    accumulate = old_btc is not None or y_old_btc is not None
    nbytes = _lib.check(lib.st2_adain_conv1d_fused_ex_scratch_bytes(B, T, Cin, Cout, k), "fused_ex_scratch_bytes")
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev())
    _lib.check(lib.st2_adain_conv1d_fused_ex(_lib.ptr(xd), _lib.ptr(hd), _lib.ptr(ad), _lib.ACT[act], C.c_float(slope),
                                             _lib.ptr(wd), _lib.ptr(bd), _lib.ptr(rd), _lib.ptr(od), _lib.ptr(y), _lib.ptr(hn),
                                             _lib.ptr(cn), _lib.ptr(scratch), B, T, Cin, Cout, k, padding, dilation,
                                             C.c_float(scale), int(accumulate), int(x16), int(res16), int(old16), int(y16),
                                             int(old_in_y), _lib.PREC[precision], stream()), "adain_conv1d_fused_ex")
    torch.cuda.synchronize()
    return y.cpu().numpy(), (None if cn is None else cn.cpu().numpy())


def act_conv_transpose1d_fused_ex(x_btc, alpha, act, w, bias, res_btc, h_next, stride, padding, output_padding, slope=0.0,
                                  precision="bf16", y16=False):
    """st2_act_conv_transpose1d_fused_ex: the upsampling step, y written as fp16 (and widened) when y16."""
    lib = _lib.load()
    B, T, Cin = x_btc.shape
    _, Cout, k = w.shape
    Tout = (T - 1) * stride - 2 * padding + (k - 1) + output_padding + 1
    xd, wd = to_dev(x_btc), to_dev(w)
    ad = None if alpha is None else to_dev(alpha.reshape(-1))
    bd = None if bias is None else to_dev(bias)
    rd = None if res_btc is None else to_dev(res_btc)
    hn = None if h_next is None else to_dev(h_next)
    cn = None if h_next is None else torch.full((B, 2, Cout), float("nan"), device=dev())
    y = torch.full((B, Tout, Cout), float("nan"), device=dev())
    nbytes = _lib.check(lib.st2_act_conv_transpose1d_fused_ex_scratch_bytes(B, T, Cin, Cout, k, stride), "fused_t_ex_scratch_bytes")
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev())
    _lib.check(lib.st2_act_conv_transpose1d_fused_ex(_lib.ptr(xd), _lib.ptr(ad), _lib.ACT[act], C.c_float(slope), _lib.ptr(wd),
                                                     _lib.ptr(bd), _lib.ptr(rd), _lib.ptr(y), _lib.ptr(hn), _lib.ptr(cn),
                                                     _lib.ptr(scratch), B, T, Cin, Cout, k, stride, padding, output_padding,
                                                     int(y16), _lib.PREC[precision], stream()), "act_conv_transpose1d_fused_ex")
    torch.cuda.synchronize()
    return y.cpu().numpy(), (None if cn is None else cn.cpu().numpy())


def har_source_dev(f0_dev, lin_w, lin_b, scale, seed):
    """st2_har_source with noise drawn on the device (Philox, noise = NULL); f0 and the result stay on the device [B,S]."""
    lib = _lib.load()
    B, L2 = f0_dev.shape
    w, b = to_dev(lin_w.reshape(-1)), to_dev(lin_b.reshape(-1))
    har = torch.full((B, L2 * scale), float("nan"), device=dev())
    frames = torch.empty(B, L2, 9, device=dev())
    _lib.check(lib.st2_har_source(_lib.ptr(f0_dev), None, C.c_uint64(seed), _lib.ptr(w), _lib.ptr(b), _lib.ptr(har),
                                  _lib.ptr(frames), B, L2, scale, stream()), "har_source")
    torch.cuda.synchronize()
    return har


def noise_conv(har_dev, w, bias, h, Tout, stride, pad, y16):
    """st2_noise_conv on a device har [B,S]; w [C,1,k]; h [B,2C] or None.  Returns device tensors (y [B,Tout,C] fp32, or fp16
    without the bias when y16; coef [B,2,C] or None)."""
    lib = _lib.load()
    B, S = har_dev.shape
    Cc, _, k = w.shape
    wd, bd = to_dev(w), to_dev(bias)
    hd = None if h is None else to_dev(h)
    coef = None if h is None else torch.full((B, 2, Cc), float("nan"), device=dev())
    y = torch.full((B, Tout, Cc), float("nan"), device=dev(), dtype=torch.float16 if y16 else torch.float32)
    nbytes = _lib.check(lib.st2_noise_conv_scratch_bytes(B, Tout, Cc, k, stride), "noise_conv_scratch_bytes")
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev())
    _lib.check(lib.st2_noise_conv(_lib.ptr(har_dev), _lib.ptr(wd), _lib.ptr(bd), _lib.ptr(y), _lib.ptr(hd), _lib.ptr(coef),
                                  _lib.ptr(scratch), B, S, Tout, Cc, k, stride, pad, int(y16), stream()), "noise_conv")
    torch.cuda.synchronize()
    return y, coef


def post_hifigan(x_dev, Cc, alpha, w, bias, fast, x16):
    """st2_post_hifigan on a device x [B,S,ld_x] (fp32, or fp16 when x16) of which the first Cc channels are used; w [1,Cc,7].
    Returns the device waveform [B,S]."""
    lib = _lib.load()
    B, S, ld = x_dev.shape
    ad, wd, bd = to_dev(alpha.reshape(-1)), to_dev(w), to_dev(bias.reshape(-1))
    out = torch.full((B, S), float("nan"), device=dev())
    wsc = torch.empty(7 * Cc, device=dev())
    _lib.check(lib.st2_post_hifigan(_lib.ptr(x_dev), ld, _lib.ptr(ad), _lib.ptr(wd), _lib.ptr(bd), _lib.ptr(out), _lib.ptr(wsc),
                                    B, S, Cc, int(fast), int(x16), stream()), "post_hifigan")
    torch.cuda.synchronize()
    return out


def style_fc(s_dev, W_dev, b_dev):
    """st2_style_fc: h [B,R] = s [B,K] @ W[R,K]^T + bias, all device tensors."""
    lib = _lib.load()
    B, K = s_dev.shape
    R = W_dev.shape[0]
    h = torch.full((B, R), float("nan"), device=dev())
    _lib.check(lib.st2_style_fc(_lib.ptr(s_dev), _lib.ptr(W_dev), _lib.ptr(b_dev), _lib.ptr(h), B, R, K, stream()), "style_fc")
    torch.cuda.synchronize()
    return h
