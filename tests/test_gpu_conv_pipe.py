"""-m gpu: conv_pipe.cu and conv_fused.cu (about 45 % of the 64 x 5 s step) against the reference when every CTA runs many
tiles, with the fp16 storage types the decoder gives them.

Both kernels are persistent: CTA i walks tiles i, i + grid, i + 2 * grid, ... and carries its rings, barrier parities and
accumulator cursors from one tile to the next.  test_gpu_fused.py runs B = 3, T <= 1000 (one tile per CTA); the benchmark runs
about 68 tiles per CTA at 128 channels.  Here the layer classes of the benchmark's plan (stage 1: x16 / res16 / old16 / y16,
tile pairs, the fp16 stage sum updated in place, the ups.1 output as fp16 in 5 N passes; stage 0: 256-channel N passes and
conv_fused) run at least 5 tiles per CTA, sized from the device's SM count; the tile walk runs at its edges (one tile more
than the grid, pairs within and across utterances, the last tile of a CTA unpaired, rows ending 1 / 127 into a tile, both
sides of the PDL cutoff, one utterance over every CTA); every launch runs twice and must repeat bitwise.  A guard runs the benchmark's shape and
checks that every conv_pipe / conv_fused class of its plan is one pinned here; a whole-decoder test pins stages 0-1 at a
batch where those layers run many tiles per CTA.

Reference: test_gpu_fused.py's half-step.  Inputs the kernel stores as fp16 are made fp16-representable first, operands are
rounded as the oracle rounds them and the conv runs as a torch CPU conv1d on the rounded operands (float32 accumulation: the
products are exact); statistics are float64 two-pass.  Bars: TOL[prec] relative to the output scale, + FP16_OUT when y is
stored as fp16; AdaIN coefficients within 2 * TOL."""
import contextlib

import numpy as np
import pytest
import torch

from styletts2_lite_b200.config import DecoderConfig
from styletts2_lite_b200 import synth
from oracle import decoder_np as O
from helpers import np_inputs, rel_l2, resblock_tap_shapes, snr_db

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import gpu_util as G
    from styletts2_lite_b200 import _lib
    from styletts2_lite_b200.decoder import B200Decoder

TOL = {"bf16": 4e-3, "fp16": 6e-4}           # test_gpu_fused.py: operands one 16-bit ulp apart (Snake through cos.approx)
FP16_OUT = 2.5e-4                            # + half an fp16 ulp of the output scale when y is stored as fp16
MIN_TILES_PER_CTA = 5                        # every CTA runs at least this many tiles in the many-tile unit cases

# launches of one bf16 HiFi-GAN forward at the benchmark's shape (64 x 200) with the default dispatch, per profile category
BENCH_LAUNCHES = {"conv_pipe": 41, "conv_fused": 12, "conv_row": 47}

_CACHE = {}


@contextlib.contextmanager
def _tuning(name, value):
    _lib.set_tuning(name, value)
    try:
        yield
    finally:
        _lib.set_tuning(name, 0)


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _h(a):
    return a.astype(np.float16).astype(np.float32)


def _plan_lines(text, kind):
    """The `kind:` plan lines (conv_pipe / conv_fused) that switch "verbose" prints, as {field: int}."""
    out = []
    for line in text.splitlines():
        if line.startswith(kind + ":"):
            out.append({k: int(v) for k, v in (kv.split("=") for kv in line.split()[1:])})
    return out


def _key(kind, ln):
    """Layer class of a plan line: (kernel, Cin, Cout, taps, nres, x16, r16, o16, y16, pair, nt, phases)."""
    if kind == "conv_pipe":
        return ("pipe", ln["Cin"], ln["Cout"] // ln["phases"], ln["taps"], ln["nres"], ln["x16"], ln["r16"], ln["o16"],
                ln["y16"], ln["pair"], ln["nt"], ln["phases"])
    return ("fused", ln["Cin"], ln["Cout"], ln["taps"], ln["res"] + ln["acc"], ln["x16"], 0, 0, ln["y16"], 0, ln["ntile_n"],
            ln["phases"])


def _relmax(got, ref):
    return float(np.abs(np.nan_to_num(got, nan=np.inf) - ref).max() / np.abs(ref).max())


def _coef(y, h_next):
    """AdaIN coefficients (a, b) of y [B,C,T] for style h_next from float64 two-pass statistics."""
    C_ = y.shape[1]
    y64 = y.astype(np.float64)
    mean = y64.mean(axis=2)
    var = ((y64 - mean[:, :, None]) ** 2).mean(axis=2)
    a = (1.0 + h_next[:, :C_].astype(np.float64)) / np.sqrt(var + 1e-5)
    return np.stack([a, h_next[:, C_:].astype(np.float64) - mean * a], axis=1)


def _bits_equal(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


# ---------------------------------------------------------------- shapes and shared operands
ROWS = {256: 4000, 128: 20000, 64: 60000, 32: 120000}      # rows per utterance of stages 0-3 at the benchmark's T = 200


def _batch_for(mtiles, sms, per_cta=MIN_TILES_PER_CTA):
    """Utterances that give every CTA of a full grid at least per_cta tiles (and a quarter of them one more)."""
    return -(-(per_cta * sms + sms // 4) // mtiles)


def _operands(C_, B, T):
    """x, h, h_next, alpha, res, old of one geometry, drawn once per module run."""
    key = ("ops", C_, B, T)
    if key not in _CACHE:
        rng = np.random.default_rng([C_, B, T])
        x = (rng.standard_normal((B, C_, T), dtype=np.float32) * 1.5 + 0.3).astype(np.float32)
        h = (rng.standard_normal((B, 2 * C_)) * 0.3).astype(np.float32)
        h_next = (rng.standard_normal((B, 2 * C_)) * 0.3).astype(np.float32)
        alpha = (0.6 + 0.8 * rng.random((1, C_, 1))).astype(np.float32)
        res = rng.standard_normal((B, C_, T), dtype=np.float32)
        old = rng.standard_normal((B, C_, T), dtype=np.float32)
        _CACHE[key] = (x, h, h_next, alpha, res, old)
    return _CACHE[key]


def _weights(Cout, Cin, k, seed):
    rng = np.random.default_rng([Cout, Cin, k, seed])
    w = (rng.standard_normal((Cout, Cin, k)) / np.sqrt(Cin * k)).astype(np.float32)
    b = rng.standard_normal(Cout).astype(np.float32)
    return w, b


def _act_operand(x, h, alpha, prec, key):
    """round_operand(snake(AdaIN(x; h)), prec) as the oracle forms the conv's input, as a torch CPU tensor (cached per key)."""
    k = ("v", key, prec)
    if k not in _CACHE:
        C_ = x.shape[1]
        v = ((1 + h[:, :C_, None]) * O.instance_norm(x) + h[:, C_:, None]).astype(np.float32)
        _CACHE[k] = torch.from_numpy(O.round_operand(O.snake(v, alpha), prec))
    return _CACHE[k]


def _conv_ref(v, w, b, dil, prec):
    """Length-preserving conv1d on the rounded operands (torch CPU, float32 accumulation)."""
    k = w.shape[2]
    wo = torch.from_numpy(O.round_operand(w, prec))
    with torch.no_grad():
        return torch.nn.functional.conv1d(v, wo, torch.from_numpy(b), padding=dil * (k - 1) // 2, dilation=dil).numpy()


# ---------------------------------------------------------------- a / b. conv_pipe half-steps
def _pipe_step(name, C_, k, dil, B, T, prec, x16=0, res=None, old=None, y16=0, scale=1.0, capfd=None, kind="conv_pipe",
               no_pipe=False):
    """One AdaINResBlock1 half-step through st2_adain_conv1d_fused_ex, twice, with the plan lines.
    res: None | "fp32" | "fp16";  old: None | "y" (fp32 old values in y) | "fp16" (separate fp16 source) | "in_y" (fp16 source
    stored into the fp16 y, accumulated in place).  kind: the kernel expected to run it (its plan line is returned); no_pipe
    sets the switch that keeps conv_pipe out.  Returns (plan line, relmax, coef relmax, bitwise repeat, nan count)."""
    x, h, h_next, alpha, r, o = _operands(C_, B, T)
    if x16:
        x = _h(x)
    res_v = None if res is None else (_h(r) if res == "fp16" else r)
    old_v = None if old is None else (o if old == "y" else _h(o))
    w, b = _weights(C_, C_, k, 1 + len(name))
    v = _act_operand(x, h, alpha, prec, (C_, B, T, x16))
    ref = _conv_ref(v, w, b, dil, prec)
    if res_v is not None:
        ref += res_v
    if old_v is not None:
        ref += old_v
    if scale != 1.0:
        ref *= np.float32(scale)
    runs = []
    ctx = _tuning("no_pipe", 1) if no_pipe else contextlib.nullcontext()
    capfd.readouterr()
    with _tuning("verbose", 1), ctx:
        for _ in range(2):
            runs.append(G.adain_conv1d_fused_ex(
                G.cl(x), h, alpha, "snake", w, b, None if res_v is None else G.cl(res_v),
                None if old_v is None or old == "y" else G.cl(old_v), G.cl(old_v) if old == "y" else None, h_next,
                dil * (k - 1) // 2, dil, scale=scale, precision=prec, x16=bool(x16), res16=res == "fp16",
                old16=old in ("fp16", "in_y"), y16=bool(y16), old_in_y=old == "in_y"))
    err_text = capfd.readouterr().err
    lines = _plan_lines(err_text, kind)
    assert len(lines) == 2 and lines[0] == lines[1], err_text[-2000:]
    assert not _plan_lines(err_text, "conv_fused" if kind == "conv_pipe" else "conv_pipe")
    (y1, c1), (y2, c2) = runs
    got = G.cf(y1)
    nan = int(np.isnan(got).sum())
    err = _relmax(got, ref)
    cref = _coef(ref, h_next)
    cerr = _relmax(c1, cref)
    same = _bits_equal(y1, y2) and _bits_equal(c1, c2)
    return lines[0], err, cerr, same, nan


def _check(test, plan, err, cerr, same, nan, prec, y16, **kv):
    G.log(test, prec=prec, relmax=err, coef_relmax=cerr, repeat_bitwise=same, nan=nan, **kv, **plan)
    assert nan == 0
    assert err <= TOL[prec] + (FP16_OUT if y16 else 0.0), err
    assert cerr <= 2 * TOL[prec], cerr
    assert same, "second launch differs"


# The benchmark's conv_pipe classes (program.cuh resblock1, decoder.cu) at stage 1 (128 channels), stage 0 (256) and the one
# stage-2 conv conv_row does not take (64 channels, k = 11, two fp16 sources -> fp32 stage output): name, C, k,
# dil, x16, res, old, y16, scale, expected pair, expected nt.  conv1 reads the block input (fp32 or the fp16 stage input) or
# the fp16 running tensor and writes the fp16 intra-block tensor; conv2 adds the running tensor (fp32 for the first iteration
# of a block whose input is fp32) and writes the next running tensor, the fp16 stage sum (first block), updates it in place
# (middle block) or writes the fp32 stage output from it (last block, scale 1/3); noise_res writes the fp32 source tensor.
PIPE_CLASSES = (
    [("c128_conv1_k%d_d%d_x%d" % (k, d, x), 128, k, d, x, None, None, 1, 1.0, 0, 1)
     for k in (3, 7, 11) for d in (1, 3, 5) for x in (0, 1)] +
    [("c128_conv2_k%d" % k, 128, k, 1, 1, "fp16", None, 1, 1.0, int(k > 3), 1) for k in (3, 7, 11)] +
    [("c128_conv2_middle_k7", 128, 7, 1, 1, "fp16", "in_y", 1, 1.0, 0, 1),
     ("c128_conv2_last_k11", 128, 11, 1, 1, "fp16", "fp16", 0, 1.0 / 3.0, 0, 1),
     ("c128_noise_res_conv2_last_k7", 128, 7, 1, 1, "fp16", None, 0, 1.0, 1, 1),
     ("c256_conv1_k3_x0", 256, 3, 3, 0, None, None, 1, 1.0, 0, 2),
     ("c256_conv1_k3_x1", 256, 3, 5, 1, None, None, 1, 1.0, 0, 2),
     ("c256_conv2_k3_first", 256, 3, 1, 1, "fp32", None, 1, 1.0, 0, 2),
     ("c256_conv2_k3", 256, 3, 1, 1, "fp16", None, 1, 1.0, 0, 2),
     ("c256_conv2_k3_last", 256, 3, 1, 1, "fp16", None, 0, 1.0, 0, 2),
     ("c256_conv1_k7", 256, 7, 3, 0, None, None, 0, 1.0, 0, 2),
     ("c256_conv2_k7_acc", 256, 7, 1, 0, "fp32", "y", 0, 1.0, 0, 2),
     ("c64_conv2_last_k11", 64, 11, 1, 1, "fp16", "fp16", 0, 1.0 / 3.0, 0, 1)])


def _class_key(C_, k, x16, res, old, y16, pair, nt):
    nres = (res is not None) + (old is not None)
    return ("pipe", C_, C_, k, nres, x16, int(res == "fp16"), int(old in ("fp16", "in_y")), y16, pair, nt, 1)


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
@pytest.mark.parametrize("name,C_,k,dil,x16,res,old,y16,scale,pair,nt", PIPE_CLASSES)
def test_conv_pipe_bench_classes_many_tiles(name, C_, k, dil, x16, res, old, y16, scale, pair, nt, prec, capfd):
    sms = _sms()
    T = ROWS[C_]
    B = _batch_for(-(-T // 128), sms)
    plan, err, cerr, same, nan = _pipe_step(name, C_, k, dil, B, T, prec, x16=x16, res=res, old=old, y16=y16, scale=scale,
                                            capfd=capfd)
    _check("conv_pipe_bench_class", plan, err, cerr, same, nan, prec, y16, case=name, B=B, T=T)
    assert _key("conv_pipe", plan) == _class_key(C_, k, x16, res, old, y16, pair, nt)
    assert plan["tiles"] >= MIN_TILES_PER_CTA * plan["grid"] and plan["grid"] == sms


# ---------------------------------------------------------------- b. tile-walk edges of conv_pipe
# the tile-pair layer (128 channels, k = 7, one fp16 residual: conv2 of stage 1) unless stated otherwise
def _edge_shape(edge, sms):
    """(C, k, B, T) of a launch that hits `edge` of the tile walk tile = blockIdx.x + i * grid."""
    if edge == "tiles_grid_plus_1":                  # one CTA runs a pair, every other one a single unpaired tile
        return 128, 7, 1, sms * 128 + 60
    if edge == "mtiles_eq_grid":                     # d_mt = 0: a CTA's tiles are the same row tile of consecutive utterances
        return 128, 7, 3, sms * 128 - 37
    if edge == "mtiles_gt_grid":                     # d_b = 0: both tiles of a pair in one utterance, 5 tiles per CTA
        return 128, 7, 2, (2 * sms + sms // 2) * 128 - 50
    if edge == "mtiles_lt_grid":                     # pairs straddle utterances
        mt = sms // 3 + 1
        return 128, 7, _batch_for(mt, sms), mt * 128 - 70
    if edge == "pair_odd_even":                      # some CTAs run an odd number of tiles (last one unpaired), some even
        mt = sms + sms // 3 + 1
        return 128, 7, 4, mt * 128 - 9
    if edge == "t_mod_1":
        return 128, 11, _batch_for(40, sms), 39 * 128 + 1
    if edge == "t_mod_127":
        return 128, 11, _batch_for(40, sms), 39 * 128 + 127
    if edge == "pdl_at_cutoff":                      # num_tiles = 16 * sms: still launched with programmatic dependent launch
        return 32, 3, 1, 16 * sms * 128
    if edge == "pdl_above_cutoff":
        return 32, 3, 1, 16 * sms * 128 + 1
    if edge == "long_utterance":                     # one utterance whose statistics come from every CTA
        return 128, 7, 1, 8 * sms * 128 + 77
    raise ValueError(edge)


EDGES = ["tiles_grid_plus_1", "mtiles_eq_grid", "mtiles_gt_grid", "mtiles_lt_grid", "pair_odd_even", "t_mod_1", "t_mod_127",
         "pdl_at_cutoff", "pdl_above_cutoff", "long_utterance"]


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
@pytest.mark.parametrize("edge", EDGES)
def test_conv_pipe_tile_walk_edges(edge, prec, capfd):
    sms = _sms()
    C_, k, B, T = _edge_shape(edge, sms)
    plan, err, cerr, same, nan = _pipe_step(edge, C_, k, 1, B, T, prec, x16=1, res="fp16", y16=1, capfd=capfd)
    grid, tiles, mt = plan["grid"], plan["tiles"], plan["mtiles"]
    _check("conv_pipe_tile_walk_edge", plan, err, cerr, same, nan, prec, 1, edge=edge, B=B, T=T,
           tiles_per_cta_min=tiles // grid, tiles_per_cta_max=-(-tiles // grid))
    assert grid == min(sms, tiles) and tiles == B * mt
    assert plan["pair"] == int(C_ == 128) and plan["r16"] == 1 and plan["x16"] == 1 and plan["y16"] == 1
    assert plan["pdl"] == int(tiles <= 16 * sms)
    if edge == "tiles_grid_plus_1":
        assert tiles == grid + 1
    elif edge == "mtiles_eq_grid":
        assert mt == grid and tiles == 3 * grid
    elif edge == "mtiles_gt_grid":
        assert mt > grid and B * mt >= MIN_TILES_PER_CTA * grid
    elif edge == "mtiles_lt_grid":
        assert mt < grid and tiles >= MIN_TILES_PER_CTA * grid
    elif edge == "pair_odd_even":
        assert tiles % grid != 0 and tiles // grid >= 4              # CTAs with q and q + 1 tiles: one count odd, one even
    elif edge in ("t_mod_1", "t_mod_127"):
        assert T % 128 == (1 if edge == "t_mod_1" else 127) and tiles >= MIN_TILES_PER_CTA * grid
    elif edge == "pdl_at_cutoff":
        assert tiles == 16 * sms and plan["pdl"] == 1
    elif edge == "pdl_above_cutoff":
        assert tiles == 16 * sms + 1 and plan["pdl"] == 0
    else:
        assert B == 1 and tiles >= 8 * grid


# ---------------------------------------------------------------- c. conv_fused at many tiles
# stride-1 classes of stage 0 that conv_pipe leaves to conv_fused (256 channels, k = 11; k = 7 with one residual), and one
# conv_pipe class forced onto conv_fused: name, C, k, dil, res, old, scale, no_pipe
FUSED_CLASSES = [
    ("c256_k11_d1", 256, 11, 1, None, None, 1.0, False), ("c256_k11_d3", 256, 11, 3, None, None, 1.0, False),
    ("c256_k11_d5", 256, 11, 5, None, None, 1.0, False), ("c256_k11_res", 256, 11, 1, "fp32", None, 1.0, False),
    ("c256_k11_res_acc_last", 256, 11, 1, "fp32", "y", 1.0 / 3.0, False), ("c256_k7_res", 256, 7, 1, "fp32", None, 1.0, False),
    ("c128_k7_res_no_pipe", 128, 7, 1, "fp32", None, 1.0, True),
]


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
@pytest.mark.parametrize("name,C_,k,dil,res,old,scale,no_pipe", FUSED_CLASSES)
def test_conv_fused_many_tiles(name, C_, k, dil, res, old, scale, no_pipe, prec, capfd):
    sms = _sms()
    T = ROWS[C_]
    B = _batch_for(-(-T // 128), sms)
    plan, err, cerr, same, nan = _pipe_step(name, C_, k, dil, B, T, prec, res=res, old=old, scale=scale, capfd=capfd,
                                            kind="conv_fused", no_pipe=no_pipe)
    _check("conv_fused_many_tiles", plan, err, cerr, same, nan, prec, 0, case=name, B=B, T=T, no_pipe=no_pipe)
    assert plan["tiles"] >= MIN_TILES_PER_CTA * plan["grid"] and plan["grid"] == sms
    assert plan["phases"] == 1 and plan["res"] == int(res is not None) and plan["acc"] == int(old is not None)


# ConvTranspose1d of the generator: ups.0 (512 -> 256, stride 10) on conv_fused, the TileIter over (b, phase, row tile) with a
# grid that is not a multiple of phases * mtiles; ups.1-3 on conv_pipe with the fp16 stage input (ups.1: 640 columns in 5 N
# passes).  name, Cin, Cout, k, stride, pad, out_pad, Tin (0: chosen from the SM count), y16, kernel, nt
UPS_CLASSES = [
    ("ups0", 512, 256, 20, 10, 5, 0, 0, 0, "conv_fused", 1),
    ("ups1_y16", 256, 128, 10, 5, 3, 1, 4000, 1, "conv_pipe", 5),
    ("ups2_y16", 128, 64, 6, 3, 2, 1, 20000, 1, "conv_pipe", 1),
    ("ups3_y16", 64, 32, 4, 2, 1, 0, 60000, 1, "conv_pipe", 1),
]


def _ups_key(Cin, Cout, k, stride, y16, kind, nt):
    return ("pipe" if kind == "conv_pipe" else "fused", Cin, Cout, k // stride, 1, 0, 0, 0, y16, 0, nt, stride)


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
@pytest.mark.parametrize("name,Cin,Cout,k,stride,pad,opad,Tin,y16,kind,nt", UPS_CLASSES)
def test_ups_many_tiles(name, Cin, Cout, k, stride, pad, opad, Tin, y16, kind, nt, prec, capfd):
    sms = _sms()
    if Tin == 0:                                     # ups.0: 4 row tiles per phase unless the grid is a multiple of 40
        Tin = 400 if sms % 40 else 300
    Tout = (Tin - 1) * stride - 2 * pad + k + opad
    M = (Tout - 1 + pad) // stride + 1
    mt = -(-M // 128)
    B = _batch_for(mt * (stride if kind == "conv_fused" else 1), sms)
    rng = np.random.default_rng([Cin, Cout, k, Tin])
    x = (rng.standard_normal((B, Cin, Tin), dtype=np.float32) * 1.2).astype(np.float32)
    alpha = (0.6 + 0.8 * rng.random((1, Cin, 1))).astype(np.float32)
    w = (rng.standard_normal((Cin, Cout, k)) / np.sqrt(Cin * k / stride)).astype(np.float32)
    b = rng.standard_normal(Cout).astype(np.float32)
    h_next = (rng.standard_normal((B, 2 * Cout)) * 0.3).astype(np.float32)
    res = rng.standard_normal((B, Cout, Tout), dtype=np.float32)
    v = torch.from_numpy(O.round_operand(O.snake(x, alpha), prec))
    with torch.no_grad():
        ref = torch.nn.functional.conv_transpose1d(v, torch.from_numpy(O.round_operand(w, prec)), torch.from_numpy(b),
                                                   stride=stride, padding=pad, output_padding=opad).numpy()
    ref += res
    capfd.readouterr()
    runs = []
    with _tuning("verbose", 1):
        for _ in range(2):
            runs.append(G.act_conv_transpose1d_fused_ex(G.cl(x), alpha, "snake", w, b, G.cl(res), h_next, stride, pad, opad,
                                                        precision=prec, y16=bool(y16)))
    text = capfd.readouterr().err
    lines = _plan_lines(text, kind)
    assert len(lines) == 2 and lines[0] == lines[1], text[-2000:]
    assert not _plan_lines(text, "conv_fused" if kind == "conv_pipe" else "conv_pipe")
    plan = lines[0]
    (y1, c1), (y2, c2) = runs
    got = G.cf(y1)
    assert got.shape == ref.shape
    nan = int(np.isnan(got).sum())
    err = _relmax(got, ref)
    cerr = _relmax(c1, _coef(ref, h_next))
    same = _bits_equal(y1, y2) and _bits_equal(c1, c2)
    _check("ups_many_tiles", plan, err, cerr, same, nan, prec, y16, case=name, B=B, Tin=Tin)
    assert _key(kind, plan) == _ups_key(Cin, Cout, k, stride, y16, kind, nt)
    assert plan["tiles"] >= MIN_TILES_PER_CTA * plan["grid"] and plan["grid"] == sms
    if kind == "conv_fused":
        assert plan["mtiles"] == mt and plan["tiles"] == B * stride * mt
        assert plan["grid"] % (stride * mt) != 0
    else:
        assert plan["mtiles"] == mt and plan["tiles"] == B * mt


# ---------------------------------------------------------------- e. the benchmark's plan is what the unit cases pin
def _covered_keys():
    keys = {_class_key(C_, k, x16, res, old, y16, pair, nt) for (_, C_, k, _d, x16, res, old, y16, _s, pair, nt) in PIPE_CLASSES}
    keys |= {("fused", C_, C_, k, (res is not None) + (old is not None), 0, 0, 0, 0, 0, 1, 1)
             for (_, C_, k, _d, res, old, _s, _np) in FUSED_CLASSES}
    keys |= {_ups_key(Cin, Cout, k, s, y16, kind, nt) for (_, Cin, Cout, k, s, _p, _o, _t, y16, kind, nt) in UPS_CLASSES}
    return keys


def _decoder():
    if "model" not in _CACHE:
        cfg = DecoderConfig.hifigan()
        m = B200Decoder(cfg, "bf16")
        m.load_state_dict(synth.make_state_dict(cfg, 0, True))
        _CACHE["model"] = m.to("cuda").eval()
    return _CACHE["model"]


def test_bench_shape_plan_is_covered(capfd):
    """64 x 200 eager bf16 forward, default dispatch, switch "verbose" on: every conv_pipe / conv_fused launch belongs to a layer
    class pinned above, the plan has tile pairs, an fp16 stage sum updated in place and an fp16 ups output, and the per-kernel
    launch counts are BENCH_LAUNCHES (a change of the dispatch shows up here before it silently leaves a class unpinned)."""
    cfg = DecoderConfig.hifigan()
    m = _decoder()
    inp = {k: v.cuda() for k, v in synth.make_inputs(64, 200, seed=1002, cfg=cfg, with_noise=False).items()}
    capfd.readouterr()
    m.set_profiling(True)
    try:
        with _tuning("verbose", 1), torch.no_grad():
            m(inp["asr"], inp["F0_curve"], inp["N"], inp["s"], seed=3, precision="bf16")
        torch.cuda.synchronize()
        prof = m.get_profile()
    finally:
        m.set_profiling(False)
    text = capfd.readouterr().err
    seen = {}
    for kind in ("conv_pipe", "conv_fused"):
        for ln in _plan_lines(text, kind):
            key = _key(kind, ln)
            seen.setdefault(key, []).append(ln["tiles"] / ln["grid"])
    launches = {k: prof[k]["launches"] for k in BENCH_LAUNCHES}
    covered = _covered_keys()
    G.log("bench_shape_plan", launches=launches, classes=[list(k) + [min(v), len(v)] for k, v in sorted(seen.items())],
          uncovered=[list(k) for k in sorted(set(seen) - covered)])
    assert set(seen) <= covered, sorted(set(seen) - covered)
    assert any(k[0] == "pipe" and k[9] == 1 for k in seen)                      # tile pairs
    assert any(k[0] == "pipe" and k[7] == 1 for k in seen)                      # fp16 stage sum
    assert any(k[0] == "pipe" and k[11] > 1 and k[8] == 1 for k in seen)        # fp16 ups output
    assert sum(len(v) for k, v in seen.items() if k[0] == "pipe") == launches["conv_pipe"]
    assert sum(len(v) for k, v in seen.items() if k[0] == "fused") == launches["conv_fused"]
    assert launches == BENCH_LAUNCHES


# ---------------------------------------------------------------- f. stages 0-1 of the whole decoder at a many-tile batch
class _Keep(dict):
    """A taps dict for the torch port that keeps only the named taps."""

    def __init__(self, names):
        super().__init__()
        self.names = set(names)

    def __setitem__(self, k, v):
        if k in self.names:
            super().__setitem__(k, v)


def test_default_dispatch_stage0_stage1_taps_vs_torch_port():
    """B = 16, T = 200, no switch: stage 1 runs 16 x 157 = 2,512 conv_pipe tiles per conv (about 17 per CTA), stage 0 about
    3.5 per CTA.  Every stage-0 / stage-1 tap <= 1e-2 relative L2 and the waveform >= 40 dB, per utterance, against the torch
    port on the CPU with the same noise tape, on the first, a middle and the last utterance."""
    from oracle import decoder_torch as OT
    cfg = DecoderConfig.hifigan()
    B, T, sub = 16, 200, (0, 7, 15)
    m = _decoder()
    inp = np_inputs(B, T, 1301, cfg)
    names = resblock_tap_shapes(T, stages=(0, 1))
    bufs = {n: m.set_tap(n, B, rows, C_) for n, (rows, C_) in names.items()}
    try:
        t = {k: torch.from_numpy(v).cuda() for k, v in inp.items()}
        with torch.no_grad():
            out = m(t["asr"], t["F0_curve"], t["N"], t["s"], noise=t["noise"], precision="bf16")
        torch.cuda.synchronize()
        got = {n: G.cf(buf[list(sub)].cpu().numpy()) for n, buf in bufs.items()}
    finally:
        m.clear_taps()
    out = out.cpu().numpy()
    del bufs
    if "W" not in _CACHE:
        _CACHE["W"] = OT.TorchWeights(synth.make_state_dict(cfg, 0, True))
    taps = _Keep(names)
    idx = list(sub)
    ti = {k: torch.from_numpy(v[idx]) for k, v in inp.items()}
    with torch.no_grad():
        ref = OT.decoder_forward(_CACHE["W"], cfg, ti["asr"], ti["F0_curve"], ti["N"], ti["s"], ti["noise"], taps=taps).numpy()
    res = {(n, b): rel_l2(taps[n][i].numpy(), a[i]) for n, a in got.items() for i, b in enumerate(sub)}
    worst = max(res, key=res.get)
    per = [snr_db(ref[i], out[b]) for i, b in enumerate(sub)]
    G.log("conv_pipe_default_taps_B16_T200", taps=len(names), utterances=list(sub), worst_tap=worst[0],
          worst_utterance=worst[1], worst_rel_l2=res[worst], worst_utterance_db=min(per))
    assert len(taps) == len(names)
    for key, v in res.items():
        assert v <= 1e-2, (key, v)
    assert min(per) >= 40.0
