"""-m gpu: the kernels of the 64 x 5 s hifigan forward outside the resblock convolutions, in the variants the benchmark
launches, against float64 references of the same operation.

- noise_conv_kernel (generator.noise_convs[i]) at the four stage geometries, fp32 and fp16 (bias-free) output, and the AdaIN
  coefficients of its output from the kernel's (sum, sumsq) tile partials;
- post_hifigan_kernel (Snake -> conv_post -> tanh), exact and FAST (__sinf / __fdividef), fp32 and fp16 input;
- har_source_kernel on device noise (Philox4x32-10 + Box-Muller), against a numpy restatement of the draw;
- style_fc_kernel (all AdaIN fc layers in one launch), including style_dim up to 1024;
- a guard on the launch counts of the source branch and the tail at the benchmark's shape.

Every kernel runs the full batch (the benchmark's grid); the float64 reference is computed for the first, a middle and the last
utterance.  Every launch runs twice and must repeat bitwise.  Bars are a-priori rounding bounds per element (u = 2^-24):
  conv of n terms plus a bias:  (n + 1) * u * (|b| + sum |w * x|)       (fp32 FMA chain, then the bias add)
  fp16 store:                    + one fp16 ulp of the value
and the approximate intrinsics use CUDA's documented error bounds, named where they are used."""
import dataclasses

import numpy as np
import pytest
import torch

from styletts2_lite_b200.config import DecoderConfig, param_specs
from styletts2_lite_b200 import synth
from oracle import decoder_np as O

if torch.cuda.is_available():
    import gpu_util as G
    from styletts2_lite_b200.decoder import B200Decoder

U = 2.0 ** -24
_CACHE = {}


def SUB(B):
    """The utterances the reference is computed for: the first, a middle and the last."""
    return sorted({0, B // 2, B - 1})


def _sd(wseed, perturb):
    """The tensors of make_state_dict(hifigan, wseed, perturb) these tests read (the full dict is dropped)."""
    key = ("sd", wseed, perturb)
    if key not in _CACHE:
        sd = synth.make_state_dict(DecoderConfig.hifigan(), wseed, perturb)
        _CACHE[key] = {k: v.numpy().copy() for k, v in sd.items()
                       if "noise_convs." in k or "m_source." in k or ("noise_res." in k and ".adain1.0.fc." in k)}
    return _CACHE[key]


def _twice(fn):
    """Run a launch twice; the outputs (tuples of device tensors or None) must match bitwise."""
    a, b = fn(), fn()
    for x, y in zip(a if isinstance(a, tuple) else (a,), b if isinstance(b, tuple) else (b,)):
        if x is not None:
            assert torch.equal(x, y), "second launch differs"
    return a


# ---------------------------------------------------------------- Philox4x32-10 + Box-Muller, restated in numpy
_M0, _M1, _W0, _W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
_MASK = 0xFFFFFFFF


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Random123's Philox4x32-10 on uint64 arrays holding 32-bit words."""
    c = [np.asarray(x, np.uint64) & _MASK for x in (c0, c1, c2, c3)]
    k0, k1 = np.uint64(k0), np.uint64(k1)
    for _ in range(10):
        p0, p1 = np.uint64(_M0) * c[0], np.uint64(_M1) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & np.uint64(_MASK), (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & np.uint64(_MASK)]
        k0, k1 = (k0 + np.uint64(_W0)) & np.uint64(_MASK), (k1 + np.uint64(_W1)) & np.uint64(_MASK)
    return c


def device_noise(seed, b, S):
    """The 9 noise values har_source_kernel draws for samples (b, 0..S-1) of a batch with S samples per utterance:
    counter (idx_lo, idx_hi, r, 0x5354), idx = b * S + n, key = seed; u = ((float)a + 0.5f) * 2^-32 clamped to [1e-12, 1];
    z = sqrt(-2 log u1) * (cos, sin)(2 pi u2).  fp32 steps are emulated exactly; log and sincos in float64.
    Returns (z [S,9] float64, r [S,9] float64, u1 [S,9] float32)."""
    idx = np.uint64(b) * np.uint64(S) + np.arange(S, dtype=np.uint64)
    k0, k1 = seed & _MASK, (seed >> 32) & _MASK
    z, rr, uu = [], [], []
    f32 = np.float32
    for r in range(3):
        x = philox4x32_10(idx & np.uint64(_MASK), idx >> np.uint64(32), np.full(S, r, np.uint64), np.full(S, 0x5354, np.uint64),
                          k0, k1)
        for a, bb in ((x[0], x[1]), (x[2], x[3])):
            u1 = (a.astype(f32) + f32(0.5)) * f32(2.3283064365386963e-10)
            u2 = (bb.astype(f32) + f32(0.5)) * f32(2.3283064365386963e-10)
            u1 = np.minimum(np.maximum(u1, f32(1e-12)), f32(1.0))
            rad = np.sqrt(-2.0 * np.log(u1.astype(np.float64)))
            th = 2.0 * np.pi * u2.astype(np.float64)
            z += [rad * np.cos(th), rad * np.sin(th)]
            rr += [rad, rad]
            uu += [u1, u1]
    return np.stack(z[:9], 1), np.stack(rr[:9], 1), np.stack(uu[:9], 1)


def test_philox_restatement_known_answers():
    """The numpy Philox4x32-10 against Random123's published known-answer vectors (CPU only)."""
    kat = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
           ((_MASK,) * 4, (_MASK, _MASK), (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
           ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
            (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]
    for ctr, key, want in kat:
        got = tuple(int(v[0]) for v in philox4x32_10(*[np.array([c], np.uint64) for c in ctr], *key))
        assert got == want, (ctr, key, [hex(v) for v in got])


def test_fma32_emulation():
    """_fma32 is a correctly rounded fp32 fused multiply-add, including the float64 double-rounding cases (CPU only)."""
    rng = np.random.default_rng(0)
    a = rng.standard_normal(200000).astype(np.float32)
    b = rng.standard_normal(200000).astype(np.float32)
    c = rng.standard_normal(200000).astype(np.float32)
    # c = -(a*b) rounded to fp32 plus a few ulps: results whose float64 sum lands on an fp32 midpoint are common here
    c[::2] = -(a[::2] * b[::2]) + np.spacing(a[::2] * b[::2]) * rng.integers(-3, 4, 100000)
    from fractions import Fraction
    got = _fma32(a, b, c)
    for i in range(0, 200000, 997):
        exact = Fraction(float(a[i])) * Fraction(float(b[i])) + Fraction(float(c[i]))
        lo = np.float32(float(exact))
        cand = [np.nextafter(lo, np.float32(-np.inf)), lo, np.nextafter(lo, np.float32(np.inf))]
        best = min(cand, key=lambda v: (abs(Fraction(float(v)) - exact), int(np.float32(v).view(np.uint32)) & 1))
        assert got[i] == best, (i, got[i], best)


# ---------------------------------------------------------------- 1. noise_conv
STAGES = [(256, 60, 30, 15), (128, 12, 6, 3), (64, 4, 2, 1), (32, 1, 1, 0)]     # C, k, stride, pad (hifigan stages 0-3)


def _har(B, T):
    """The real harmonic source of synth.make_inputs(B, T) F0 (device noise, seed 7) on the device, and its host copy."""
    key = ("har", B, T)
    if key not in _CACHE:
        cfg = DecoderConfig.hifigan()
        sd = _sd(0, True)
        f0 = G.to_dev(synth.make_inputs(B, T, seed=1500 + B, cfg=cfg, with_noise=False)["F0_curve"].numpy())
        har = G.har_source_dev(f0, sd["generator.m_source.l_linear.weight"], sd["generator.m_source.l_linear.bias"],
                               cfg.upsample_scale, 7)
        _CACHE[key] = har
    return _CACHE[key]


def _noise_conv_ref(har_b, w, bias, Tout, stride, pad):
    """float64 Conv1d(1 -> C) of one utterance: (y [Tout,C], sum |w * x| [Tout,C])."""
    C_, _, k = w.shape
    S = har_b.shape[0]
    need = (Tout - 1) * stride + k
    hp = np.zeros(need, np.float64)
    seg = har_b.astype(np.float64)[:max(0, min(S, need - pad))]
    hp[pad:pad + seg.shape[0]] = seg
    win = np.lib.stride_tricks.sliding_window_view(hp, k)[::stride][:Tout]            # [Tout, k]
    w2 = w[:, 0, :].astype(np.float64).T                                               # [k, C]
    return win @ w2 + bias.astype(np.float64), np.abs(win) @ np.abs(w2)


def _check_noise_conv(stage, B, T, wseed, perturb, y16):
    cfg = DecoderConfig.hifigan()
    C_, k, stride, pad = STAGES[stage]
    sd = _sd(wseed, perturb)
    w = sd["generator.noise_convs.%d.weight" % stage]
    bias = sd["generator.noise_convs.%d.bias" % stage]
    s = synth.make_inputs(B, T, seed=1600 + B, cfg=cfg, with_noise=False)["s"].numpy()
    fw, fb = sd["generator.noise_res.%d.adain1.0.fc.weight" % stage], sd["generator.noise_res.%d.adain1.0.fc.bias" % stage]
    h = (s @ fw.T + fb).astype(np.float32)
    har = _har(B, T)
    S = har.shape[1]
    Tout = (S + 2 * pad - k) // stride + 1
    assert Tout == 2 * T * int(np.prod(cfg.upsample_rates[:stage + 1]))
    y_d, coef_d = _twice(lambda: G.noise_conv(har, w, bias, h, Tout, stride, pad, y16))
    sub = SUB(B)
    y = y_d[sub].float().cpu().numpy().astype(np.float64)
    coef = coef_d[sub].cpu().numpy().astype(np.float64)
    har_h = har[sub].cpu().numpy()
    b64 = bias.astype(np.float64)
    worst = dict(y=0.0, a=0.0, z=0.0)
    for i, b in enumerate(sub):
        y64, mag = _noise_conv_ref(har_h[i], w, bias, Tout, stride, pad)
        if y16:
            e_y = np.spacing(np.abs(y64 - b64).astype(np.float16)).astype(np.float64) + k * U * mag
            err = np.abs(y[i] - (y64 - b64))
        else:
            e_y = (k + 1) * U * (np.abs(b64) + mag)
            err = np.abs(y[i] - y64)
        worst["y"] = max(worst["y"], float((err / e_y).max()))
        assert (err <= e_y).all(), ("y", b, float((err / e_y).max()))
        m64 = y64.mean(0)
        sd64 = np.sqrt(((y64 - m64) ** 2).mean(0))
        gamma, beta = h[b, :C_].astype(np.float64), h[b, C_:].astype(np.float64)
        a64 = (1.0 + gamma) / np.sqrt(sd64 ** 2 + 1e-5)
        a, bb = coef[i, 0], coef[i, 1]
        ra = np.abs(a / a64 - 1.0)
        worst["a"] = max(worst["a"], float(ra.max()))
        assert (ra <= 1e-5).all(), ("rstd", b, int(ra.argmax()), float(ra.max()), float(np.abs(m64 / sd64)[ra.argmax()]))
        # normalised output a * stored + b against (1+gamma) * (y - mean) / std + beta: the error of the stored value, a mean
        # error as large as the 1e-5 the coefficients allow (in units of std), and the fp32 rounding of b and of a * stored
        z = a * y[i] + bb
        z64 = a64 * (y64 - m64) + beta
        e_z = np.abs(a) * e_y + 1e-5 * np.abs(a64) * (np.abs(y64 - m64) + sd64) + 2 * U * (np.abs(bb) + np.abs(a * y[i]))
        rz = np.abs(z - z64) / e_z
        worst["z"] = max(worst["z"], float(rz.max()))
        assert (rz <= 1).all(), ("normalised", b, float(rz.max()))
    G.log("noise_conv", stage=stage, B=B, T=T, w=[wseed, perturb], y16=y16, y_over_bar=worst["y"], rstd_rel=worst["a"],
          z_over_bar=worst["z"])


@pytest.mark.gpu
@pytest.mark.parametrize("y16", [0, 1])
@pytest.mark.parametrize("wseed,perturb", [(0, True), (3, False)])
@pytest.mark.parametrize("stage", [0, 1, 2, 3])
def test_noise_conv_bench_shape(stage, wseed, perturb, y16):
    """B = 64, T = 200 (Tout = 4,000 / 20,000 / 60,000 / 120,000): y, the fp16 bias-free store and the AdaIN coefficients."""
    _check_noise_conv(stage, 64, 200, wseed, perturb, y16)


@pytest.mark.gpu
@pytest.mark.parametrize("y16", [0, 1])
@pytest.mark.parametrize("B,T", [(3, 128), (3, 2), (1, 200), (65, 200)])
@pytest.mark.parametrize("stage", [0, 1, 2, 3])
def test_noise_conv_edges(stage, B, T, y16):
    """T = 128: Tout a multiple of the tile at stages 0, 1 and 3; T = 2: one partial tile (stages 0-2) and two (stage 3);
    B = 1 and B = 65."""
    _check_noise_conv(stage, B, T, 0, True, y16)


# ---------------------------------------------------------------- 2. post_hifigan
# FAST bounds used (CUDA C Programming Guide, intrinsic functions): __sinf(x) has an absolute error of at most 2^-21.41 for
# x in [-pi, pi] and "larger otherwise"; outside that range the bar adds the fp32 rounding of the reduction of x to
# revolutions, |x| * 2^-23.  __fdividef(x, y) has a maximum error of 2 ulp for 2^-126 <= |y| <= 2^126.
# The exact path: sinf has a maximum error of 2 ulp, tanhf of 2 ulp; 1.f / a is correctly rounded.
def _snake_ref_and_bound(x, alpha, fast):
    """float64 Snake of x [..,C] and a bound on the kernel's fp32 Snake per element."""
    al = alpha.astype(np.float64)
    u = al * x
    s = np.sin(u)
    snake = x + s * s / al
    au = np.abs(u)
    if fast:
        ds = 2.0 ** -21.41 + au * U + au * 2 * U
        rcp = 2 * 2 * U
    else:
        ds = au * U + 2 * U
        rcp = U
    ds = np.minimum(ds, 2.0)
    e = (2 * np.abs(s) * ds + ds * ds) / np.abs(al) + (rcp + 2 * U) * s * s / np.abs(al) + U * np.abs(snake)
    return snake, e


def _post_ref(x, alpha, w, bias, fast):
    """float64 tanh(conv_post(snake(x))) of one utterance x [S,C] and the bound on the kernel's error per sample."""
    S, C_ = x.shape
    sn, e_sn = _snake_ref_and_bound(x.astype(np.float64), alpha.reshape(-1), fast)
    pad = lambda a: np.concatenate([np.zeros((3, C_)), a, np.zeros((3, C_))])       # noqa: E731
    sn, e_sn = pad(sn), pad(e_sn)
    w2 = w[0].astype(np.float64)                                                    # [C, 7]
    acc = np.full(S, float(bias[0]))
    mag = np.full(S, abs(float(bias[0])))
    prop = np.zeros(S)
    for k in range(7):
        acc += sn[k:k + S] @ w2[:, k]
        mag += np.abs(sn[k:k + S]) @ np.abs(w2[:, k])
        prop += e_sn[k:k + S] @ np.abs(w2[:, k])
    out = np.tanh(acc)
    bound = prop + (7 * C_ + 1) * U * mag + 2 * U
    return out, 2 * bound                     # first-order bound, doubled for the second-order terms it drops


def _post_inputs(B, S, C_, ld, seed, x16):
    """x [B,S,ld] on the device with the amplitude of a stage-3 output (N(0, 2), 1 % of the values at |alpha * x| up to 20);
    the ld - C pad columns hold NaN, which the kernel must not read."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    rng = np.random.default_rng(seed)
    alpha = (0.2 + 1.3 * rng.random(C_)).astype(np.float32)
    w = (rng.standard_normal((1, C_, 7)) * 0.05).astype(np.float32)
    bias = np.array([0.01], np.float32)
    x = torch.randn(B, S, C_, generator=g, device="cuda") * 2.0
    big = torch.rand(B, S, C_, generator=g, device="cuda") < 0.01
    x = torch.where(big, (torch.rand(B, S, C_, generator=g, device="cuda") * 40 - 20) / G.to_dev(alpha), x)
    xd = torch.full((B, S, ld), float("nan"), device="cuda", dtype=torch.float16 if x16 else torch.float32)
    xd[:, :, :C_] = x.to(xd.dtype)
    return xd, alpha, w, bias


def _check_post(B, S, C_, ld, fast, x16, seed):
    xd, alpha, w, bias = _post_inputs(B, S, C_, ld, seed, x16)
    out_d = _twice(lambda: G.post_hifigan(xd, C_, alpha, w, bias, fast, x16))
    assert torch.isfinite(out_d).all()
    sub = SUB(B)
    out = out_d[sub].cpu().numpy().astype(np.float64)
    xs = xd[sub][:, :, :C_].float().cpu().numpy()
    worst, maxarg = 0.0, 0.0
    for i, b in enumerate(sub):
        ref, bound = _post_ref(xs[i], alpha, w, bias, fast)
        r = np.abs(out[i] - ref) / bound
        worst = max(worst, float(r.max()))
        maxarg = max(maxarg, float(np.abs(xs[i] * alpha).max()))
        assert (r <= 1).all(), (b, int(r.argmax()), float(r.max()))
        for edge in (slice(0, 3), slice(S - 3, S)):                                # the zero-padded samples at each end
            assert (np.abs(out[i][edge] - ref[edge]) <= bound[edge]).all()
    G.log("post_hifigan", B=B, S=S, C=C_, ld=ld, fast=fast, x16=x16, err_over_bar=worst, max_alpha_x=maxarg)
    return maxarg


@pytest.mark.gpu
@pytest.mark.parametrize("fast,x16", [(0, 0), (1, 0), (1, 1)])
def test_post_hifigan_bench_shape(fast, x16):
    """B = 64, S = 120,000 (not a multiple of the 256-sample tile), C = 32."""
    maxarg = _check_post(64, 120000, 32, 32, fast, x16, 11 + fast + x16)
    assert maxarg >= 15.0


@pytest.mark.gpu
@pytest.mark.parametrize("fast,x16", [(0, 0), (1, 0), (1, 1)])
@pytest.mark.parametrize("B,S,C_,ld", [(3, 5000, 64, 64), (2, 777, 32, 40), (2, 512, 64, 72)])
def test_post_hifigan_edges(B, S, C_, ld, fast, x16):
    """C = 64 (shared memory above 48 KB), ld_x > C, S a multiple of the tile and not."""
    _check_post(B, S, C_, ld, fast, x16, 100 + S + C_ + fast + x16)


# ---------------------------------------------------------------- 3. har_source on device noise
@pytest.mark.gpu
@pytest.mark.parametrize("seed", [0, 5, 2 ** 63 + 5])
def test_har_source_device_noise_vs_float64(seed):
    """B = 64, L2 = 400: har against the float64 source formula fed with the restated Philox / Box-Muller noise.  The SineGen
    phase is the fp32 one the kernel reads (bit-exact with oracle.sinegen_phase, test_gpu_units.py).  Bound per sample:
    sinf 2 ulp, the fp32 roundings of the chain, tanhf 2 ulp, and the noise's error from __logf (absolute 2^-21.41 on
    [0.5, 2], 3 ulp elsewhere) and __sincosf (absolute 2^-21.41 on [-pi, pi], plus |x| * 2^-23 for the reduction beyond)."""
    cfg = DecoderConfig.hifigan()
    B, T, scale = 64, 200, cfg.upsample_scale
    sd = _sd(0, True)
    lw, lb = sd["generator.m_source.l_linear.weight"].reshape(-1), sd["generator.m_source.l_linear.bias"].reshape(-1)
    f0 = synth.make_inputs(B, T, seed=1700, cfg=cfg, with_noise=False)["F0_curve"].numpy()
    f0d = G.to_dev(f0)
    har_d = _twice(lambda: G.har_source_dev(f0d, lw, lb, scale, seed))
    sub = SUB(B)
    har = har_d[sub].cpu().numpy().astype(np.float64)
    L2 = f0.shape[1]
    S = L2 * scale
    phase = O.sinegen_phase(f0[sub], scale).astype(np.float64)                       # [3,S,9]
    lw64 = np.abs(lw.astype(np.float64))
    worst, worst_abs = 0.0, 0.0
    for i, b in enumerate(sub):
        z, r, u1 = device_noise(seed, b, S)
        uv = (f0[b][np.arange(S) // scale] > 10.0).astype(np.float64)[:, None]
        namp = uv * 0.003 + (1 - uv) * 0.1 / 3
        sw = np.sin(phase[i]) * 0.1
        v = sw * uv + namp * z
        acc = v @ lw.astype(np.float64) + float(lb[0])
        ref = np.tanh(acc)
        # noise error: log error -> r error; sincos error of 2 pi u2 (< 2 pi)
        dlog = np.where(u1 >= 0.5, 2.0 ** -21.41, 3 * np.spacing(np.abs(np.log(u1.astype(np.float64))).astype(np.float32)))
        dr = np.minimum(np.sqrt(2 * dlog), 2 * dlog / np.maximum(r, 1e-30)) + 2 * U * r
        dz = dr + r * (2.0 ** -21.41 + 2 * np.pi * 4 * U) + U * r      # + the fp32 argument 2 pi u2 and its reduction
        e_v = namp * (dz + 2 * U * np.abs(z)) + 0.1 * uv * (3 * U) + 2 * U * np.abs(v)
        bound = e_v @ lw64 + 10 * U * (abs(float(lb[0])) + np.abs(v) @ lw64) + 2 * U
        err = np.abs(har[i] - ref)
        worst = max(worst, float((err / bound).max()))
        worst_abs = max(worst_abs, float(err.max()))
        assert (err <= bound).all(), (b, int((err / bound).argmax()), float((err / bound).max()))
    G.log("har_source_device_noise", seed=str(seed), err_over_bar=worst, max_abs=worst_abs)


@pytest.mark.gpu
def test_har_source_device_noise_moments_and_independence():
    """The noise the kernel draws, read back through an unvoiced source with one-hot weights (har = tanh(0.1/3 * z_h)), over
    64 utterances x 120,000 samples per harmonic: mean, std, correlation at lag 1, across utterances (b, b+1) and across
    harmonics (h, h+1), each within 5 / sqrt(N)."""
    cfg = DecoderConfig.hifigan()
    B, L2, scale = 64, 400, cfg.upsample_scale
    f0 = torch.zeros(B, L2, device="cuda")
    namp = float(np.float32(np.float32(0.1) / np.float32(3.0)))
    prev = None
    stats = []
    for h in range(9):
        w = np.zeros(9, np.float32)
        w[h] = 1.0
        har = G.har_source_dev(f0, w, np.zeros(1, np.float32), scale, 11)
        z = torch.atanh(har.double()) / namp
        N = z.numel()
        bar = 5.0 / np.sqrt(N)
        zc = z - z.mean()
        var = float((zc * zc).mean())
        mean, std = float(z.mean()), float(np.sqrt(var))
        lag1 = float((zc[:, 1:] * zc[:, :-1]).mean()) / var
        utt = float((zc[1:] * zc[:-1]).mean()) / var
        har_c = float((zc * prev).mean()) / np.sqrt(var * float((prev * prev).mean())) if prev is not None else 0.0
        stats.append(dict(h=h, mean=mean, std=std, lag1=lag1, utt=utt, prev_h=har_c))
        assert abs(mean) <= bar and abs(std - 1) <= bar / np.sqrt(2), stats[-1]
        assert abs(lag1) <= bar and abs(utt) <= bar and abs(har_c) <= bar, stats[-1]
        prev = zc
    G.log("har_source_noise_moments", N=N, bar=bar, stats=stats)


# ---------------------------------------------------------------- 4. style_fc
def _fma32(a, b, c):
    """Correctly rounded fp32 fma(a, b, c) on fp32 arrays: the product is exact in float64; the float64 sum is corrected where it
    lands on an fp32 rounding midpoint (double rounding) by the sign of its TwoSum error."""
    p = a.astype(np.float64) * b.astype(np.float64)
    c64 = c.astype(np.float64)
    t = p + c64
    bp = t - p
    err = (p - (t - bp)) + (c64 - bp)
    r = t.astype(np.float32)
    r64 = r.astype(np.float64)
    lo = np.where(r64 <= t, r, np.nextafter(r, np.float32(-np.inf)))
    hi = np.where(r64 >= t, r, np.nextafter(r, np.float32(np.inf)))
    mid = (lo != hi) & ((lo.astype(np.float64) + hi.astype(np.float64)) * 0.5 == t)
    return np.where(mid & (err > 0), hi, np.where(mid & (err < 0), lo, r))


def _fc_rows():
    return sum(shape[0] for name, shape, _ in param_specs(DecoderConfig.hifigan()) if name.endswith(".fc.weight"))


def _fc_operands(R, K):
    """W [R,K], bias [R] on the device and on the host (one set cached at a time)."""
    if _CACHE.get("fc_key") != (R, K):
        g = torch.Generator(device="cuda").manual_seed(R * 7 + K)
        W = (torch.randn(R, K, generator=g, device="cuda") / np.sqrt(K)).contiguous()
        bias = torch.randn(R, generator=g, device="cuda") * 0.1
        _CACHE["fc"] = None
        _CACHE["fc"] = (W, bias, W.cpu().numpy(), bias.cpu().numpy())
        _CACHE["fc_key"] = (R, K)
    return _CACHE["fc"]


@pytest.mark.gpu
@pytest.mark.parametrize("R", ["adain", 1001])
@pytest.mark.parametrize("K", [4, 128, 908, 1024])
@pytest.mark.parametrize("B", [1, 64, 65, 129])
def test_style_fc(B, K, R):
    """h = s @ W^T + bias: bitwise equal to the fp32 FMA chain over k = 0..K-1 then the bias add (last utterance: alone in
    the second 64-utterance block at B = 65), and within (K + 1) * u * (|b| + sum |w * s|) of float64 (first, middle, last).
    R = the decoder's AdaIN row total (42,004, not a multiple of 16) and 1,001 (a partial row quad)."""
    R = _fc_rows() if R == "adain" else R
    W, bias, Wh, bh = _fc_operands(R, K)
    s = G.to_dev(np.random.default_rng(B * 1000 + K).standard_normal((B, K)).astype(np.float32))
    h = _twice(lambda: G.style_fc(s, W, bias))
    sub = SUB(B)
    hs = h[sub].cpu().numpy()
    sh = s[sub].cpu().numpy()
    r = np.zeros(hs.shape)
    for r0 in range(0, R, 4096):                   # float64 in row chunks: host memory stays small at R x K = 42,004 x 1,024
        Wc = Wh[r0:r0 + 4096].astype(np.float64)
        ref = sh.astype(np.float64) @ Wc.T + bh[r0:r0 + 4096]
        bound = (K + 1) * U * (np.abs(bh[r0:r0 + 4096]) + np.abs(sh).astype(np.float64) @ np.abs(Wc).T)
        r[:, r0:r0 + 4096] = np.abs(hs[:, r0:r0 + 4096] - ref) / bound
    assert (r <= 1).all(), float(r.max())
    acc = np.zeros(R, np.float32)
    last = sh[-1]
    for k in range(K):
        acc = _fma32(Wh[:, k], np.full(R, last[k], np.float32), acc)
    chain = acc + bh
    mism = int((chain != hs[-1]).sum())
    G.log("style_fc", B=B, K=K, R=R, err_over_bar=float(r.max()), chain_mismatches=mism)
    assert mism == 0


@pytest.mark.gpu
def test_decoder_style_dim_1024():
    """A decoder created with style_dim = 1024 (the largest st2_decoder_create accepts) runs a small fp32 forward: finite and
    within 1e-4 of the numpy oracle, as smoke() checks the default decoder."""
    cfg = dataclasses.replace(DecoderConfig.hifigan(), style_dim=1024)
    sd = synth.make_state_dict(cfg, 0, True)
    m = B200Decoder(cfg, "fp32")
    m.load_state_dict(sd)
    m = m.to("cuda").eval()
    inp = synth.make_inputs(2, 4, seed=1234, cfg=cfg)
    t = {k: v.cuda() for k, v in inp.items()}
    with torch.no_grad():
        out = m(t["asr"], t["F0_curve"], t["N"], t["s"], noise=t["noise"])
    torch.cuda.synchronize()
    out = out.cpu().numpy()
    ref = O.decoder_forward({k: v.numpy() for k, v in sd.items()}, cfg,
                            *(inp[k].numpy() for k in ("asr", "F0_curve", "N", "s", "noise")))
    err = float(np.abs(out - ref).max())
    G.log("decoder_style_dim_1024", maxabs=err)
    assert np.isfinite(out).all()
    assert err <= 1e-4


# ---------------------------------------------------------------- 5. guard
# launches of one bf16 HiFi-GAN forward at the benchmark's shape (64 x 200), per profile category: source = the SineGen
# frames + harmonic source pair and the four noise_convs; post = conv_post's kernel
BENCH_LAUNCHES = {"source": 5, "post": 1}


@pytest.mark.gpu
def test_bench_shape_source_and_tail_launches():
    """A new kernel in the source branch or the tail shows up here before it runs unpinned."""
    cfg = DecoderConfig.hifigan()
    m = B200Decoder(cfg, "bf16")
    m.load_state_dict(synth.make_state_dict(cfg, 0, True))
    m = m.to("cuda").eval()
    inp = {k: v.cuda() for k, v in synth.make_inputs(64, 200, seed=1002, cfg=cfg, with_noise=False).items()}
    m.set_profiling(True)
    try:
        with torch.no_grad():
            m(inp["asr"], inp["F0_curve"], inp["N"], inp["s"], seed=3, precision="bf16")
        torch.cuda.synchronize()
        prof = m.get_profile()
    finally:
        m.set_profiling(False)
    launches = {k: prof[k]["launches"] for k in BENCH_LAUNCHES}
    G.log("bench_shape_source_tail", launches=launches)
    assert launches == BENCH_LAUNCHES
