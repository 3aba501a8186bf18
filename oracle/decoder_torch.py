"""CPU port of the reference decoder on torch's own CPU kernels  --  TEST / BASELINE INFRASTRUCTURE ONLY.

The reference (Modules/hifigan.py, Modules/istftnet.py) is pure PyTorch: on a CPU its arithmetic
is ATen's oneDNN convolution, native_batch_norm, upsample_linear1d, cumsum ...  This module
restates Decoder.forward as plain functions over a flat state_dict using the SAME ATen ops, so
that `bench.py --impl reference` / `cpu_baseline` time what the reference really executes on the
host cores (the numpy oracle in decoder_np.py is ~6x slower than that and is the parity checker,
not a fair speed baseline).  tests/test_oracle.py pins it to the golden fixtures exactly like the
numpy oracle.  Nothing in styletts2_lite_b200/ imports this file.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import numpy as np
import torch
import torch.nn.functional as F


def _fold(sd, name):
    """weight_norm fold, torch._weight_norm(v, g, 0) (hifigan.py:30, 292, 317, 373, 377, 434)."""
    if name + ".weight_g" in sd:
        return torch._weight_norm(sd[name + ".weight_v"], sd[name + ".weight_g"], 0)
    return sd[name + ".weight"]


class TorchWeights:
    def __init__(self, sd: Dict[str, torch.Tensor]):
        self.sd = {k: (v if isinstance(v, torch.Tensor) else torch.from_numpy(np.asarray(v))).float() for k, v in sd.items()}
        self._w: Dict[str, torch.Tensor] = {}

    def w(self, name):
        if name not in self._w:
            self._w[name] = _fold(self.sd, name).contiguous()
        return self._w[name]

    def b(self, name):
        return self.sd.get(name + ".bias")

    def p(self, name):
        return self.sd[name]


def adain(W, name, x, s):
    """AdaIN1d.forward, hifigan.py:20-24."""
    h = F.linear(s, W.p(name + ".fc.weight"), W.p(name + ".fc.bias"))
    gamma, beta = torch.chunk(h.unsqueeze(-1), 2, dim=1)
    return (1 + gamma) * F.instance_norm(x) + beta


def snake(x, a):
    """hifigan.py:68."""
    return x + (1 / a) * (torch.sin(a * x) ** 2)


def adain_resblk1d(W, name, x, s, upsample):
    """AdainResBlk1d.forward, hifigan.py:384-403."""
    h = F.leaky_relu(adain(W, name + ".norm1", x, s), 0.2)
    if upsample:
        h = F.conv_transpose1d(h, W.w(name + ".pool"), W.b(name + ".pool"), stride=2, padding=1, output_padding=1,
                               groups=h.shape[1])
    h = F.conv1d(h, W.w(name + ".conv1"), W.b(name + ".conv1"), padding=1)
    h = F.leaky_relu(adain(W, name + ".norm2", h, s), 0.2)
    h = F.conv1d(h, W.w(name + ".conv2"), W.b(name + ".conv2"), padding=1)
    sc = F.interpolate(x, scale_factor=2, mode="nearest") if upsample else x
    if name + ".conv1x1.weight_v" in W.sd:
        sc = F.conv1d(sc, W.w(name + ".conv1x1"))
    return (h + sc) / math.sqrt(2)


def adain_resblock1(W, name, x, s, k, dil=(1, 3, 5), taps=None):
    """AdaINResBlock1.forward, hifigan.py:65-74.  taps: optional dict that receives the conv1 output (`.convs1.j`) and the
    running tensor after every iteration (`.iterj`), the names the library's debug taps use."""
    for j, d in enumerate(dil):
        xt = snake(adain(W, "%s.adain1.%d" % (name, j), x, s), W.p("%s.alpha1.%d" % (name, j)))
        xt = F.conv1d(xt, W.w("%s.convs1.%d" % (name, j)), W.b("%s.convs1.%d" % (name, j)), dilation=d,
                      padding=int((k * d - d) / 2))
        if taps is not None:
            taps["%s.convs1.%d" % (name, j)] = xt
        xt = snake(adain(W, "%s.adain2.%d" % (name, j), xt, s), W.p("%s.alpha2.%d" % (name, j)))
        xt = F.conv1d(xt, W.w("%s.convs2.%d" % (name, j)), W.b("%s.convs2.%d" % (name, j)), padding=int((k - 1) / 2))
        x = xt + x
        if taps is not None:
            taps["%s.iter%d" % (name, j)] = x
    return x


def source_module(W, f0_curve, scale, noise):
    """SineGen + SourceModuleHnNSF, hifigan.py:117-157, 189-218, 254-264 (noise = the randn_like draw)."""
    f0 = F.interpolate(f0_curve[:, None], scale_factor=float(scale), mode="nearest").transpose(1, 2)   # [B,S,1]
    fn = f0 * torch.arange(1, 10, dtype=torch.float32, device=f0.device).view(1, 1, 9)
    rad = (fn / 24000) % 1
    rad = F.interpolate(rad.transpose(1, 2), scale_factor=1 / scale, mode="linear").transpose(1, 2)
    phase = torch.cumsum(rad, dim=1) * 2 * np.pi
    phase = F.interpolate(phase.transpose(1, 2) * scale, scale_factor=float(scale), mode="linear").transpose(1, 2)
    sine = torch.sin(phase) * 0.1
    uv = (f0 > 10).float()
    noise_amp = uv * 0.003 + (1 - uv) * 0.1 / 3
    sine = sine * uv + noise_amp * noise
    har = torch.tanh(F.linear(sine, W.p("generator.m_source.l_linear.weight"), W.p("generator.m_source.l_linear.bias")))
    return har.transpose(1, 2)


def decoder_forward(W, cfg, asr, F0_curve, N, s, noise, taps=None):
    """Decoder.forward (eval), hifigan.py:446-475 / istftnet.py:692-721 with Generator.forward inlined.
    taps: optional dict filled with intermediate tensors [B, C, T] under the library's tap names."""
    with torch.no_grad():
        F0 = F.conv1d(F0_curve[:, None], W.w("F0_conv"), W.b("F0_conv"), stride=2, padding=1)
        Nn = F.conv1d(N[:, None], W.w("N_conv"), W.b("N_conv"), stride=2, padding=1)
        x = adain_resblk1d(W, "encode", torch.cat([asr, F0, Nn], 1), s, False)
        asr_res = F.conv1d(asr, W.w("asr_res.0"), W.b("asr_res.0"))
        if taps is not None:
            taps["encode"] = x
        for i in range(4):
            x = adain_resblk1d(W, "decode.%d" % i, torch.cat([x, asr_res, F0, Nn], 1), s, i == 3)
            if taps is not None:
                taps["decode.%d" % i] = x
        har = source_module(W, F0_curve, cfg.upsample_scale, noise)
        istft = cfg.is_istft
        if istft:
            n_fft, hop = cfg.gen_istft_n_fft, cfg.gen_istft_hop_size
            wav = F.pad(har[:, 0, :].unsqueeze(1), (n_fft // 2, n_fft // 2), mode="replicate")
            re = F.conv1d(wav, W.p("generator.stft.weight_forward_real"), stride=hop)
            im = F.conv1d(wav, W.p("generator.stft.weight_forward_imag"), stride=hop)
            mag = torch.sqrt(re ** 2 + im ** 2 + 1e-14)
            ph = torch.atan2(im, re)
            ph[(im == 0) & (re < 0)] = torch.pi
            har = torch.cat([mag, ph], 1)
        nk = len(cfg.resblock_kernel_sizes)
        for i in range(cfg.num_stages):
            x = F.leaky_relu(x, 0.1) if istft else snake(x, W.p("generator.alphas.%d" % i))
            _, k, st, pd = cfg.noise_conv_geometry(i)
            xs = F.conv1d(har, W.w("generator.noise_convs.%d" % i), W.b("generator.noise_convs.%d" % i), stride=st, padding=pd)
            xs = adain_resblock1(W, "generator.noise_res.%d" % i, xs, s, cfg.noise_res_kernel(i), taps=taps)
            ku, u, pu, opu = cfg.ups_geometry(i)
            x = F.conv_transpose1d(x, W.w("generator.ups.%d" % i), W.b("generator.ups.%d" % i), stride=u, padding=pu,
                                   output_padding=opu)
            if istft and i == cfg.num_stages - 1:
                x = F.pad(x, (1, 0), mode="reflect")
            x = x + xs
            if taps is not None:
                taps["generator.stage%d.in" % i] = x
            acc = None
            for j, kr in enumerate(cfg.resblock_kernel_sizes):
                r = adain_resblock1(W, "generator.resblocks.%d" % (i * nk + j), x, s, kr, cfg.resblock_dilation_sizes[j], taps=taps)
                acc = r if acc is None else acc + r
            x = acc / nk
            if taps is not None:
                taps["generator.stage%d.out" % i] = x
        if not istft:
            x = snake(x, W.p("generator.alphas.%d" % cfg.num_stages))
            return torch.tanh(F.conv1d(x, W.w("generator.conv_post"), W.b("generator.conv_post"), padding=3))
        x = F.conv1d(F.leaky_relu(x), W.w("generator.conv_post"), W.b("generator.conv_post"), padding=3)
        bins = n_fft // 2 + 1
        spec, phase = torch.exp(x[:, :bins]), torch.sin(x[:, bins:])
        r = F.conv_transpose1d(spec * torch.cos(phase), W.p("generator.stft.weight_backward_real"), stride=hop)
        im_ = F.conv_transpose1d(spec * torch.sin(phase), W.p("generator.stft.weight_backward_imag"), stride=hop)
        return (r - im_)[..., n_fft // 2: -(n_fft // 2)]
