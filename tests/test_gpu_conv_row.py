"""-m gpu: conv_row.cu (the 32- and 64-channel AdaINResBlock1 convolutions, the largest kernel of the 64 x 5 s step) against the
reference, in the scheduling states the benchmark's plan produces.

The decoder picks conv_row only when a conv has at least 4 macro tiles per SM, so the reference fixtures (B <= 2) run on
conv_pipe by default.  Switch "row_always" drops that threshold; every whole-decoder test here that means to run conv_row
asserts the number of conv_row launches it saw, so a later change of the dispatch cannot quietly turn it back into a
conv_pipe test.  At unit level, st2_adain_conv1d_row is driven at shapes built from the device's SM count so that the
planner's tile split (tq macro tiles per CTA, the first tr CTAs one more, J statistics slots per CTA) hits its edges: CTAs that
hold partials of up to 8 utterances, the last CTA one tile short, grids smaller than the device, a one-row last macro tile and
one 60 s utterance over every CTA.  st2_adain_conv1d_row_pair chains two launches as AdaINResBlock1 does, the second
computing its AdaIN coefficients from the first one's partials.

Bars: BASELINE.json (waveform SNR >= 40 dB, every layer relative L2 <= 1e-2) for the decoder, the bounds of
test_gpu_fused.py's conv_row unit test for the units."""
import contextlib

import numpy as np
import pytest
import torch

from styletts2_lite_b200.config import DecoderConfig
from styletts2_lite_b200 import synth
from oracle import decoder_np as O
from helpers import golden, np_inputs, rel_l2, resblock_tap_shapes, snr_db

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import gpu_util as G
    from styletts2_lite_b200 import _lib
    from styletts2_lite_b200.decoder import B200Decoder

# conv_row launches of one HiFi-GAN forward when every 32 / 64-channel AdaINResBlock1 conv runs on it: the default plan at the
# benchmark shape (64 x 200) and the forced plan at the fixture shapes
ROW_LAUNCHES = 47

TOL = {"bf16": 4e-3, "fp16": 6e-4}           # test_gpu_fused.py: operands one 16-bit ulp apart (Snake through cos.approx)
FP16_OUT = 2.5e-4                            # + half an fp16 ulp of the output scale when y is stored as fp16

_CACHE = {}


def _decoder(cfg, wseed=0, perturb=True):
    key = (cfg.type, wseed, perturb)
    if key not in _CACHE:
        m = B200Decoder(cfg, "bf16")
        m.load_state_dict(synth.make_state_dict(cfg, wseed, perturb))
        _CACHE[key] = m.to("cuda").eval()
    return _CACHE[key]


@contextlib.contextmanager
def _tuning(name, value):
    _lib.set_tuning(name, value)
    try:
        yield
    finally:
        _lib.set_tuning(name, 0)


def _row_always(on=True):
    return _tuning("row_always", 1) if on else contextlib.nullcontext()


def _forward(m, inp, prec, noise=True, seed=None):
    """Eager forward with the per-launch profile on; returns (waveform on the device, conv_row launches)."""
    t = {k: (v if torch.is_tensor(v) else torch.from_numpy(v)).cuda() for k, v in inp.items()}
    m.set_profiling(True)
    try:
        with torch.no_grad():
            out = m(t["asr"], t["F0_curve"], t["N"], t["s"], noise=t["noise"] if noise else None, seed=seed, precision=prec)
        torch.cuda.synchronize()
        n_row = m.get_profile()["conv_row"]["launches"]
    finally:
        m.set_profiling(False)
    return out, n_row


def _port(inp, utterances, taps=None):
    """oracle/decoder_torch.py (the torch port of the reference, pinned to its waveforms by tests/test_oracle.py) on the CPU
    for some utterances of a batch: every op is per utterance, so they are the rows of the full batch's result.  (On the GPU
    the port drifts from the reference with length, 41 dB at 3 s on a B200, too close to the bar to measure against.)"""
    from oracle import decoder_torch as OT
    cfg = DecoderConfig.hifigan()
    if "W" not in _CACHE:
        _CACHE["W"] = OT.TorchWeights(synth.make_state_dict(cfg, 0, True))
    idx = list(utterances)
    t = {k: (v if torch.is_tensor(v) else torch.from_numpy(v))[idx] for k, v in inp.items()}
    with torch.no_grad():
        return OT.decoder_forward(_CACHE["W"], cfg, t["asr"], t["F0_curve"], t["N"], t["s"], t["noise"], taps=taps).numpy()


# ---------------------------------------------------------------- the switch and the module's caches
def test_row_always_switch_replans_eager_and_graph():
    """Flipping a switch through _lib.set_tuning changes the plan of the next forward, eager and captured: the graph captured
    before the flip is not replayed (it would run conv_pipe again) and the workspace is sized for the new plan."""
    cfg = DecoderConfig.hifigan()
    m = _decoder(cfg)
    inp = {k: v.cuda() for k, v in synth.make_inputs(1, 30, seed=130, cfg=cfg, with_noise=False).items()}

    def both():
        eager, n_row = _forward(m, inp, "bf16", noise=False, seed=21)
        with torch.no_grad():
            graph = m(inp["asr"], inp["F0_curve"], inp["N"], inp["s"], seed=21, precision="bf16", cuda_graph=True)
        torch.cuda.synchronize()
        return eager, graph, n_row
    e0, g0, n0 = both()
    with _row_always():
        e1, g1, n1 = both()
    e2, g2, n2 = both()
    G.log("row_always_replan", launches_default=n0, launches_forced=n1, snr_between_db=snr_db(e0.cpu().numpy(), e1.cpu().numpy()))
    assert n0 == 0 and n2 == 0 and n1 == ROW_LAUNCHES
    assert torch.equal(g0, e0) and torch.equal(g1, e1) and torch.equal(g2, e2)
    assert not torch.equal(e1, e0)                 # another kernel: other rounding
    assert torch.equal(e2, e0)


# ---------------------------------------------------------------- a. reference goldens with conv_row forced
GOLDEN_CASES = [
    # fixture, B, T, weight seed, input seed, perturbed weights
    ("hifigan_B2_T5_w0_i1001", 2, 5, 0, 1001, True),
    ("hifigan_B1_T120_w0_i1001", 1, 120, 0, 1001, True),
    ("hifigan_B1_T120_w3_i1007_plain", 1, 120, 3, 1007, False),
    ("hifigan_B1_T203_w0_i1009", 1, 203, 0, 1009, True),
    ("hifigan_B1_T400_w0_i1003", 1, 400, 0, 1003, True),
]


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
@pytest.mark.parametrize("name,B,T,ws,iseed,perturb", GOLDEN_CASES)
def test_conv_row_forced_vs_reference_goldens(name, B, T, ws, iseed, perturb, prec):
    """Every 32 / 64-channel resblock conv on conv_row: SNR >= 40 dB against the unmodified reference's waveform (the default
    plan, mostly conv_pipe at these sizes, is logged beside it)."""
    cfg = DecoderConfig.hifigan()
    g = golden(name + ".npz")["out"]
    m = _decoder(cfg, ws, perturb)
    inp = np_inputs(B, T, iseed, cfg)
    base, n_base = _forward(m, inp, prec)
    with _row_always():
        out, n_row = _forward(m, inp, prec)
    out = out.cpu().numpy()
    snr, snr_base = snr_db(g, out), snr_db(g, base.cpu().numpy())
    G.log("conv_row_forced_vs_golden", fixture=name, prec=prec, snr_db=snr, snr_default_db=snr_base, launches=n_row,
          launches_default=n_base, maxabs=float(np.abs(out - g).max()))
    assert out.shape == g.shape
    assert n_row == ROW_LAUNCHES
    assert snr >= 40.0


# ---------------------------------------------------------------- b. every layer with conv_row forced, 3 s
def test_bf16_every_resblock_tap_at_3s_on_conv_row():
    """test_gpu_decoder.py::test_bf16_every_resblock_tap_at_3s with every 32 / 64-channel resblock conv on conv_row: each tap
    <= 1e-2 relative L2 against the torch CPU port of the reference, waveform >= 40 dB."""
    cfg = DecoderConfig.hifigan()
    T = 120
    m = _decoder(cfg)
    inp = np_inputs(1, T, 1001, cfg)
    names = resblock_tap_shapes(T)
    bufs = {n: m.set_tap(n, 1, rows, C_) for n, (rows, C_) in names.items()}
    try:
        with _row_always():
            out, n_row = _forward(m, inp, "bf16")
    finally:
        got = {n: G.cf(buf.cpu().numpy()) for n, buf in bufs.items()}
        m.clear_taps()
    taps = {}
    ref = _port(inp, [0], taps)
    res = {n: rel_l2(taps[n].numpy(), a) for n, a in got.items()}
    worst = max(res, key=res.get)
    snr = snr_db(ref, out.cpu().numpy())
    G.log("conv_row_forced_every_tap_T120", taps=len(res), worst_tap=worst, worst_rel_l2=res[worst], snr_db=snr, launches=n_row)
    assert n_row == ROW_LAUNCHES
    for n, v in res.items():
        assert v <= 1e-2, (n, v)
    assert snr >= 40.0


# ---------------------------------------------------------------- c / d. the default dispatch against the torch port
def test_default_dispatch_stage2_stage3_taps_vs_torch_port():
    """B = 9, T = 120, no switch: the 64- and 32-channel stages have enough macro tiles for the default plan to pick conv_row.
    Every stage-2 / stage-3 tap (conv1 outputs, running tensors, stage input / output) <= 1e-2 relative L2 and the waveform
    >= 40 dB, per utterance, against the torch port with the same noise tape, on the first, a middle and the last utterance.
    (Stages 0-1 are pinned at B = 1.)"""
    cfg = DecoderConfig.hifigan()
    B, T, sub = 9, 120, (0, 4, 8)
    m = _decoder(cfg)
    inp = np_inputs(B, T, 1201, cfg)
    names = resblock_tap_shapes(T, stages=(2, 3))
    bufs = {n: m.set_tap(n, B, rows, C_) for n, (rows, C_) in names.items()}
    try:
        out, n_row = _forward(m, inp, "bf16")
        got = {n: G.cf(buf[list(sub)].cpu().numpy()) for n, buf in bufs.items()}
    finally:
        m.clear_taps()
    out = out.cpu().numpy()
    taps = {}
    ref = _port(inp, sub, taps)
    res = {(n, b): rel_l2(taps[n][i].numpy(), a[i]) for n, a in got.items() for i, b in enumerate(sub)}
    worst = max(res, key=res.get)
    per = [snr_db(ref[i], out[b]) for i, b in enumerate(sub)]
    G.log("conv_row_default_taps_B9_T120", taps=len(names), utterances=list(sub), worst_tap=worst[0], worst_utterance=worst[1],
          worst_rel_l2=res[worst], worst_utterance_db=min(per), launches=n_row)
    assert n_row == ROW_LAUNCHES
    for key, v in res.items():
        assert v <= 1e-2, (key, v)
    assert min(per) >= 40.0


BENCH_SUBSET = tuple(range(0, 64, 9))            # 8 of the 64 utterances, the first and the last among them


@pytest.fixture(scope="module")
def bench_shape_port():
    """The benchmark's workload (64 x 5 s) with an explicit noise tape, and the torch port's waveforms of BENCH_SUBSET."""
    inp = synth.make_inputs(64, 200, seed=1002, cfg=DecoderConfig.hifigan(), with_noise=True)
    return inp, _port(inp, BENCH_SUBSET)


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
def test_bench_shape_vs_torch_port(prec, bench_shape_port):
    """64 x 200, default dispatch (the kernel plan bench.py times) with ROW_LAUNCHES conv_row launches: >= 40 dB against the
    torch port over BENCH_SUBSET and for each of its utterances; every utterance finite."""
    inp, ref = bench_shape_port
    m = _decoder(DecoderConfig.hifigan())
    out, n_row = _forward(m, inp, prec)
    out = out.cpu().numpy()
    per = {b: snr_db(ref[i], out[b]) for i, b in enumerate(BENCH_SUBSET)}
    worst = min(per, key=per.get)
    snr = snr_db(ref, out[list(BENCH_SUBSET)])
    G.log("conv_row_bench_shape_vs_port", prec=prec, snr_db=snr, worst_utterance=worst, worst_utterance_db=per[worst],
          launches=n_row)
    assert np.isfinite(out).all()
    assert n_row == ROW_LAUNCHES
    assert snr >= 40.0 and per[worst] >= 40.0


# ---------------------------------------------------------------- 4. scheduling edges of one launch
def _ref(x, h, alpha, w, b, res, old, pad, dil, scale, prec):
    """One half-step of AdaINResBlock1 in the oracle (test_gpu_fused.py's reference)."""
    C_ = x.shape[1]
    v = ((1 + h[:, :C_, None]) * O.instance_norm(x) + h[:, C_:, None]).astype(np.float32)
    y = O.conv1d(O.snake(v, alpha), w, b, padding=pad, dilation=dil, operand=prec)
    if res is not None:
        y = y + res
    if old is not None:
        y = y + old
    return (y * np.float32(scale)).astype(np.float32)


def _coef(y, h_next):
    """AdaIN coefficients (a, b) of y for style h_next from float64 two-pass statistics."""
    C_ = y.shape[1]
    y64 = y.astype(np.float64)
    mean = y64.mean(axis=2)
    var = ((y64 - mean[:, :, None]) ** 2).mean(axis=2)
    a = (1.0 + h_next[:, :C_].astype(np.float64)) / np.sqrt(var + 1e-5)
    return np.stack([a, h_next[:, C_:].astype(np.float64) - mean * a], axis=1)


def _h(a):
    return a.astype(np.float16).astype(np.float32)


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _sub(C_, k, nres):
    """The planner's macro tile (128-row MMA sub-tiles) for these layers: everything 32-channel takes 4; at 64 channels the
    operand buffers leave room for 2 (k = 3, or k = 7 without fp16 sources), 1 otherwise."""
    if C_ == 32:
        return 4
    return 2 if (k == 3 and nres < 2) or (k == 7 and nres == 0) else 1


def _row_plan(B, T, sub, sms):
    """row_plan's tile split (conv_row.cu): grid, tq macro tiles per CTA with the first tr CTAs one more, J slots per CTA."""
    mmt = -(-T // (sub * 128))
    nt = B * mmt
    grid = min(sms, 160, nt)
    tq, tr = divmod(nt, grid)
    return {"sub": sub, "mmt": mmt, "grid": grid, "tq": tq, "tr": tr, "J": -(-(tq + 1) // mmt) + 1}


def _edge_shape(edge, C_, sub, sms):
    """(B, T) of a launch that hits `edge` of the tile split."""
    R, g = sub * 128, min(sms, 160)
    jmax = 2048 // (2 * C_ * 4)                      # statistics slots whose coefficient table fits the kernel's 2 KB
    if edge == "tr_zero":                            # every CTA the same number (2) of macro tiles; odd mmt: CTAs straddle
        nt = 2 * g
        B = next(b for b in range(2, nt + 1) if nt % b == 0 and (nt // b) % 2 == 1)
        return B, (nt // B) * R - R // 3
    if edge == "tr_last":                            # tr = grid - 1: only the last CTA owns one tile less
        for q in range(1, 8):
            nt = q * g + g - 1
            B = next((b for b in range(2, 64) if nt % b == 0), None)
            if B:
                return B, (nt // B) * R - R // 2
        raise AssertionError("no shape with tr = grid - 1")
    if edge == "small_grid":                         # fewer macro tiles than SMs: grid = B * mmt
        return 3, (g // 6) * R - 5
    if edge == "j_at_limit":                         # one tile per utterance, tq + 1 = J - 1 utterances per CTA
        return (jmax - 2) * g + g // 2, min(R - 3, 130)
    if edge == "j_above_limit":
        return (jmax - 1) * g + g // 3, min(R - 3, 100)
    if edge == "tail_one_row":                       # every utterance ends one row into a macro tile
        return g - 1, 2 * R + 1
    raise ValueError(edge)


def _verbose_lines(text):
    return [dict(kv.split("=") for kv in l.split()[1:]) for l in text.splitlines() if l.startswith("conv_row:")]


EDGES = ["tr_zero", "tr_last", "small_grid", "j_at_limit", "j_above_limit", "tail_one_row"]
EDGE_K = {"tr_zero": (3, 3), "tr_last": (7, 1), "small_grid": (3, 5), "j_at_limit": (3, 1), "j_above_limit": (7, 3),
          "tail_one_row": (3, 1)}


@pytest.mark.parametrize("sources", ["none", "res_old"])
@pytest.mark.parametrize("prec", ["bf16", "fp16"])
@pytest.mark.parametrize("C_", [32, 64])
@pytest.mark.parametrize("edge", EDGES)
def test_conv_row_tile_split_edges_vs_oracle(edge, C_, prec, sources, capfd):
    k, dil = EDGE_K[edge]
    if C_ == 64:
        k = 3                                        # 64-channel k = 7 with two fp16 sources runs 1-sub-tile macro tiles
    use_src = sources == "res_old"
    sub = _sub(C_, k, 2 if use_src else 0)
    sms = _sms()
    B, T = _edge_shape(edge, C_, sub, sms)
    plan = _row_plan(B, T, sub, sms)
    rng = np.random.default_rng([EDGES.index(edge), C_, len(prec), len(sources)])
    x = (rng.standard_normal((B, C_, T)) * 1.5 + 0.3).astype(np.float32)
    x16 = y16 = use_src
    if x16:
        x = _h(x)
    h = (rng.standard_normal((B, 2 * C_)) * 0.3).astype(np.float32)
    h_next = (rng.standard_normal((B, 2 * C_)) * 0.3).astype(np.float32)
    alpha = (0.6 + 0.8 * rng.random((1, C_, 1))).astype(np.float32)
    w = (rng.standard_normal((C_, C_, k)) / np.sqrt(C_ * k)).astype(np.float32)
    b = rng.standard_normal(C_).astype(np.float32)
    res = _h(rng.standard_normal((B, C_, T)).astype(np.float32)) if use_src else None
    old = _h(rng.standard_normal((B, C_, T)).astype(np.float32)) if use_src else None
    pad = dil * (k - 1) // 2
    scale = 1.0 / 3.0 if use_src else 1.0
    capfd.readouterr()
    with _tuning("row_sub", sub), _tuning("verbose", 1):
        got, coef = G.adain_conv1d_row(G.cl(x), h, alpha, w, b, None if res is None else G.cl(res),
                                       None if old is None else G.cl(old), h_next, pad, dil, scale=scale, precision=prec,
                                       x16=x16, y16=y16)
    lines = _verbose_lines(capfd.readouterr().err)
    assert len(lines) == 1, lines
    seen = {key: int(lines[0][key]) for key in plan}
    got = G.cf(got)
    ref = _ref(x, h, alpha, w, b, res, old, pad, dil, scale, prec)
    nan = int(np.isnan(got).sum())
    err = float(np.abs(np.nan_to_num(got) - ref).max() / np.abs(ref).max())
    cref = _coef(ref, h_next)
    cerr = float(np.abs(np.nan_to_num(coef) - cref).max() / np.abs(cref).max())
    G.log("conv_row_tile_split_edge", edge=edge, C=C_, prec=prec, sources=sources, B=B, T=T, k=k, dil=dil, relmax=err,
          coef_relmax=cerr, nan=nan, **seen)
    assert seen == plan
    if edge == "tr_zero":
        assert plan["tr"] == 0 and plan["tq"] >= 2
    elif edge == "tr_last":
        assert plan["tr"] == plan["grid"] - 1
    elif edge == "small_grid":
        assert plan["grid"] == B * plan["mmt"] < sms
    elif edge == "j_at_limit":
        assert plan["J"] == 2048 // (8 * C_) and plan["tq"] >= 2
    elif edge == "j_above_limit":
        assert plan["J"] == 2048 // (8 * C_) + 1
    else:
        assert T % (sub * 128) == 1
    assert nan == 0
    assert err <= TOL[prec] + (FP16_OUT if y16 else 0.0)
    assert cerr <= 2 * TOL[prec]


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
def test_conv_row_one_60s_utterance_over_every_cta(prec, capfd):
    """C = 32, B = 1, T = 1,440,000 (60 s at the last stage's rate): one utterance's statistics summed over the partials of
    every CTA.  Reference: the oracle's fp32 AdaIN and Snake, operands rounded like its conv, the conv itself in float64."""
    C_, k, dil, B, T = 32, 3, 1, 1, 1_440_000
    sms = _sms()
    plan = _row_plan(B, T, 4, sms)
    rng = np.random.default_rng(60)
    x = _h((rng.standard_normal((B, C_, T)) * 1.5 + 0.3).astype(np.float32))
    h = (rng.standard_normal((B, 2 * C_)) * 0.3).astype(np.float32)
    h_next = (rng.standard_normal((B, 2 * C_)) * 0.3).astype(np.float32)
    alpha = (0.6 + 0.8 * rng.random((1, C_, 1))).astype(np.float32)
    w = (rng.standard_normal((C_, C_, k)) / np.sqrt(C_ * k)).astype(np.float32)
    b = rng.standard_normal(C_).astype(np.float32)
    res = _h(rng.standard_normal((B, C_, T)).astype(np.float32))
    capfd.readouterr()
    with _tuning("row_sub", 4), _tuning("verbose", 1):
        got, coef = G.adain_conv1d_row(G.cl(x), h, alpha, w, b, G.cl(res), None, h_next, 1, dil, precision=prec)
    lines = _verbose_lines(capfd.readouterr().err)
    got = G.cf(got)
    v = O.snake(((1 + h[:, :C_, None]) * O.instance_norm(x) + h[:, C_:, None]).astype(np.float32), alpha)
    vo = torch.from_numpy(O.round_operand(v, prec)).double()
    wo = torch.from_numpy(O.round_operand(w, prec)).double()
    ref = (torch.nn.functional.conv1d(vo, wo, torch.from_numpy(b).double(), padding=1, dilation=dil).numpy()
           + res).astype(np.float32)
    err = float(np.abs(np.nan_to_num(got) - ref).max() / np.abs(ref).max())
    cref = _coef(ref, h_next)
    cerr = float(np.abs(np.nan_to_num(coef) - cref).max() / np.abs(cref).max())
    G.log("conv_row_60s", prec=prec, relmax=err, coef_relmax=cerr, **plan)
    assert len(lines) == 1 and {key: int(lines[0][key]) for key in plan} == plan
    assert plan["grid"] == min(sms, 160) and plan["tq"] >= 10
    assert int(np.isnan(got).sum()) == 0
    assert err <= TOL[prec] + FP16_OUT
    assert cerr <= 2 * TOL[prec]


# ---------------------------------------------------------------- two chained launches: in-kernel AdaIN coefficients
PAIR_CASES = [
    # name, C, (k1, dil1), (k2, dil2), mmt, tq: CTAs hold partials of up to tq / mmt + 2 utterances
    ("eight_utterances_per_cta", 32, (3, 3), (3, 1), 2, 12),
    ("j_at_limit_c64", 64, (3, 5), (3, 1), 1, 2),
    ("j_above_limit", 32, (7, 1), (7, 1), 1, 7),
    ("small_grid", 32, (11, 5), (11, 1), 4, 0),
]


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
@pytest.mark.parametrize("name,C_,kd1,kd2,mmt,tq", PAIR_CASES)
def test_conv_row_pair_inline_coefficients_vs_oracle(name, C_, kd1, kd2, mmt, tq, prec, capfd):
    """y1 = step(x), y2 = step(y1) + x with the second launch computing the AdaIN coefficients of y1 from the first launch's
    per-(CTA, utterance, warp) partials when they fit its 2 KB table (J * 2 * C floats), the coefficient kernel otherwise, and
    again with switch "no_row_inline_coef".  The second step's reference starts from the kernel's own stored y1 with float64
    two-pass statistics; both runs meet the single-step bounds."""
    (k1, dil1), (k2, dil2) = kd1, kd2
    sub = _sub(C_, 3, 1)
    sms = _sms()
    g = min(sms, 160)
    R = sub * 128
    if tq == 0:
        B = 3
    else:
        B = (tq * g + g // 4) // mmt
    T = (mmt - 1) * R + R // 5
    plan = _row_plan(B, T, sub, sms)
    if tq:
        assert plan["tq"] == tq, plan
    inline_expected = plan["J"] * 2 * C_ * 4 <= 2048
    rng = np.random.default_rng([[c[0] for c in PAIR_CASES].index(name), len(prec)])
    x = _h((rng.standard_normal((B, C_, T)) * 1.5 + 0.3).astype(np.float32))
    h1, h2, h_next = ((rng.standard_normal((B, 2 * C_)) * 0.3).astype(np.float32) for _ in range(3))
    a1, a2 = ((0.6 + 0.8 * rng.random((1, C_, 1))).astype(np.float32) for _ in range(2))
    w1 = (rng.standard_normal((C_, C_, k1)) / np.sqrt(C_ * k1)).astype(np.float32)
    w2 = (rng.standard_normal((C_, C_, k2)) / np.sqrt(C_ * k2)).astype(np.float32)
    b1, b2 = (rng.standard_normal(C_).astype(np.float32) for _ in range(2))
    runs = {}
    for no_inline in (0, 1):
        capfd.readouterr()
        with _tuning("row_sub", sub), _tuning("verbose", 1), _tuning("no_row_inline_coef", no_inline):
            y1, y2, coef, inline = G.adain_conv1d_row_pair(G.cl(x), h1, a1, w1, b1, h2, a2, w2, b2, h_next, dil1, dil2,
                                                           precision=prec)
        lines = _verbose_lines(capfd.readouterr().err)
        runs[no_inline] = (G.cf(y1), G.cf(y2), coef, inline, lines)
    ref1 = _ref(x, h1, a1, w1, b1, None, None, dil1 * (k1 - 1) // 2, dil1, 1.0, prec)
    for no_inline, (y1, y2, coef, inline, lines) in runs.items():
        assert len(lines) == 2, lines
        for ln in lines:
            assert {key: int(ln[key]) for key in plan} == plan
        assert int(lines[1]["inline"]) == int(inline)
        assert inline == (inline_expected and not no_inline)
        ref2 = _ref(y1, h2, a2, w2, b2, x, None, dil2 * (k2 - 1) // 2, dil2, 1.0, prec)
        cref = _coef(ref2, h_next)
        e1 = float(np.abs(np.nan_to_num(y1) - ref1).max() / np.abs(ref1).max())
        e2 = float(np.abs(np.nan_to_num(y2) - ref2).max() / np.abs(ref2).max())
        cerr = float(np.abs(np.nan_to_num(coef) - cref).max() / np.abs(cref).max())
        G.log("conv_row_pair", case=name, prec=prec, no_row_inline_coef=no_inline, inline=inline, B=B, T=T, relmax1=e1,
              relmax2=e2, coef_relmax=cerr, **plan)
        assert e1 <= TOL[prec] + FP16_OUT
        assert e2 <= TOL[prec] + FP16_OUT, (no_inline, e2)
        assert cerr <= 2 * TOL[prec]
