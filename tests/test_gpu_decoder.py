"""-m gpu: whole-decoder parity through the drop-in module / C ABI.

fp32 path: max-abs <= 1e-4 against the golden waveforms of the unmodified reference
(BASELINE.json north_star) with the shared noise tape; per-layer taps against the oracle.
16-bit tensor-core paths: SNR >= 40 dB and per-layer relative L2 <= 1e-2."""
import numpy as np
import pytest
import torch

from styletts2_lite_b200.config import DecoderConfig
from styletts2_lite_b200 import synth
from oracle import decoder_np as O
from helpers import golden, np_inputs, np_state_dict, rel_l2, snr_db

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import gpu_util as G
    from styletts2_lite_b200 import _lib, hifigan, istftnet
    from styletts2_lite_b200.decoder import B200Decoder

_CACHE = {}


def _decoder(cfg, wseed=0, perturb=True, precision="fp32"):
    key = (cfg.type, wseed, perturb)
    if key not in _CACHE:
        m = B200Decoder(cfg, precision)
        m.load_state_dict(synth.make_state_dict(cfg, wseed, perturb))
        _CACHE[key] = m.to("cuda").eval()
    return _CACHE[key]


def _run(m, inp, precision="fp32", noise=True, seed=None):
    t = {k: torch.from_numpy(v).cuda() for k, v in inp.items()}
    with torch.no_grad():
        out = m(t["asr"], t["F0_curve"], t["N"], t["s"], noise=t["noise"] if noise else None, seed=seed,
                precision=precision)
    torch.cuda.synchronize()
    return out.cpu().numpy()


def _tap_table(m, cfg, inp, names_shapes, precision="fp32"):
    """Run with debug taps and compare each against the oracle's tap; returns {name: rel_l2}."""
    B = inp["asr"].shape[0]
    bufs = {n: m.set_tap(n, B, rows, C_) for n, (rows, C_) in names_shapes.items()}
    out = _run(m, inp, precision)
    taps = {}
    sd = np_state_dict(cfg, 0, True)
    ref = O.decoder_forward(sd, cfg, inp["asr"], inp["F0_curve"], inp["N"], inp["s"], inp["noise"], taps=taps)
    res = {}
    for n, buf in bufs.items():
        a = G.cf(buf.cpu().numpy())
        res[n] = rel_l2(taps[n], a)
    m.clear_taps()
    return out, ref, res


def test_state_dict_is_drop_in():
    m = hifigan.Decoder(dim_in=512, style_dim=128, dim_out=80, resblock_kernel_sizes=[3, 7, 11],
                        upsample_rates=[10, 5, 3, 2], upsample_initial_channel=512,
                        resblock_dilation_sizes=[[1, 3, 5]] * 3, upsample_kernel_sizes=[20, 10, 6, 4])
    assert sum(p.numel() for p in m.parameters()) == 54_289_492        # README.md:21
    assert len(m.state_dict()) == 678
    m2 = istftnet.Decoder(style_dim=128)
    assert sum(p.numel() for p in m2.parameters()) == 53_276_190
    assert len(m2.state_dict()) == 380


def test_hifigan_small_fp32_golden_and_taps():
    cfg = DecoderConfig.hifigan()
    g = golden("hifigan_B2_T5_w0_i1001.npz")
    inp = np_inputs(2, 5, 1001, cfg)
    m = _decoder(cfg)
    T = 5
    shapes = {"har_source": (600 * T, 1), "encode.conv1": (T, 1024), "encode": (T, 1024), "decode.0": (T, 1024),
              "decode.3": (2 * T, 512), "generator.noise_res.0.iter2": (20 * T, 256),
              "generator.stage0.in": (20 * T, 256), "generator.resblocks.0.iter1": (20 * T, 256),
              "generator.stage0.out": (20 * T, 256), "generator.stage1.out": (100 * T, 128),
              "generator.stage2.out": (300 * T, 64), "generator.noise_res.3.iter2": (600 * T, 32),
              "generator.stage3.out": (600 * T, 32)}
    out, ref, res = _tap_table(m, cfg, inp, shapes)
    for n, v in res.items():
        G.log("hifigan_small_tap", tap=n, rel_l2=v)
    err_g = float(np.abs(out - g["out"]).max())
    err_o = float(np.abs(out - ref).max())
    G.log("hifigan_small", maxabs_vs_golden=err_g, maxabs_vs_oracle=err_o, launches=m.last_launch_count())
    for n, v in res.items():
        assert v <= 1e-4, (n, v)
    assert err_g <= 1e-4


def test_hifigan_reference_init_fp32_golden():
    cfg = DecoderConfig.hifigan()
    g = golden("hifigan_B1_T4_w3_i1002_plain.npz")
    m = _decoder(cfg, 3, False)
    out = _run(m, np_inputs(1, 4, 1002, cfg))
    err = float(np.abs(out - g["out"]).max())
    G.log("hifigan_plain", maxabs_vs_golden=err)
    assert err <= 1e-4


def test_hifigan_cfg1_3s_fp32_golden():
    """BASELINE.json configs[0] shape: B=1, T=120 (3 s)."""
    cfg = DecoderConfig.hifigan()
    g = golden("hifigan_B1_T120_w0_i1001.npz")
    m = _decoder(cfg)
    inp = np_inputs(1, 120, 1001, cfg)
    har = m.set_tap("har_source", 1, 72000, 1)
    out = _run(m, inp)
    err_h = float(np.abs(har.cpu().numpy()[:, :, 0] - g["har_source"][:, :, 0]).max())
    m.clear_taps()
    err = float(np.abs(out - g["out"]).max())
    G.log("hifigan_cfg1", maxabs_vs_golden=err, har_source_maxabs=err_h, snr_db=snr_db(g["out"], out))
    assert err_h <= 1e-6
    assert err <= 1e-4


def test_istftnet_small_fp32_golden_and_taps():
    cfg = DecoderConfig.istftnet()
    g = golden("istftnet_B2_T5_w0_i1005.npz")
    inp = np_inputs(2, 5, 1005, cfg)
    m = _decoder(cfg)
    T = 5
    shapes = {"har_source": (600 * T, 1), "har": (120 * T + 1, 22), "decode.3": (2 * T, 512),
              "generator.noise_res.0.iter2": (20 * T, 256), "generator.stage0.out": (20 * T, 256),
              "generator.noise_res.1.iter2": (120 * T + 1, 128), "generator.stage1.in": (120 * T + 1, 128),
              "generator.stage1.out": (120 * T + 1, 128)}
    out, ref, res = _tap_table(m, cfg, inp, shapes)
    for n, v in res.items():
        G.log("istftnet_small_tap", tap=n, rel_l2=v)
    err_g = float(np.abs(out - g["out"]).max())
    G.log("istftnet_small", maxabs_vs_golden=err_g, maxabs_vs_oracle=float(np.abs(out - ref).max()))
    for n, v in res.items():
        assert v <= 1e-4, (n, v)
    assert err_g <= 1e-4


def test_batch_independence_and_determinism():
    """Every op is per-utterance (SURVEY 8(e)): element b of a batch equals the B=1 run."""
    cfg = DecoderConfig.hifigan()
    m = _decoder(cfg)
    inp = np_inputs(3, 6, 1010, cfg)
    full = _run(m, inp)
    again = _run(m, inp)
    assert np.array_equal(full, again)
    one = _run(m, {k: v[1:2] for k, v in inp.items()})
    assert np.abs(one[0] - full[1]).max() <= 1e-6


def test_device_noise_seeded():
    cfg = DecoderConfig.hifigan()
    m = _decoder(cfg)
    inp = np_inputs(1, 6, 1011, cfg)
    a = _run(m, inp, noise=False, seed=123)
    b = _run(m, inp, noise=False, seed=123)
    c = _run(m, inp, noise=False, seed=124)
    assert np.array_equal(a, b) and not np.array_equal(a, c)
    assert np.isfinite(a).all() and np.abs(a).max() <= 1.0


def test_error_behaviour():
    cfg = DecoderConfig.hifigan()
    m = _decoder(cfg)
    x = torch.zeros(1, 512, 4, device="cuda")
    f = torch.zeros(1, 8, device="cuda")
    s = torch.zeros(1, 128, device="cuda")
    with pytest.raises(ValueError):
        m(x, f[:, :7], f, s)
    with pytest.raises(_lib.St2Error):
        m(x.cpu(), f.cpu(), f.cpu(), s.cpu())
    m.train(True)
    with pytest.raises(RuntimeError):
        m(x, f, f, s)
    m.train(False)
    # C ABI: forward before finalize, and too-small workspace
    import ctypes as C
    lib = _lib.load()
    h = C.c_void_p()
    cc = _lib.St2Config.from_config(cfg)
    assert lib.st2_decoder_create(C.byref(cc), C.byref(h)) == 0
    out = torch.zeros(1, 1, 2400, device="cuda")
    ws = torch.zeros(1024, dtype=torch.uint8, device="cuda")
    rc = lib.st2_decoder_forward(h, _lib.ptr(x), _lib.ptr(f), _lib.ptr(f), _lib.ptr(s), None, 0, _lib.ptr(out), 1, 4, 0,
                                 _lib.ptr(ws), ws.numel(), None)
    assert rc == -2 and b"finalize" in lib.st2_last_error()
    lib.st2_decoder_destroy(h)
    rc = lib.st2_decoder_forward(m._handle, _lib.ptr(x), _lib.ptr(f), _lib.ptr(f), _lib.ptr(s), None, 0, _lib.ptr(out), 1, 4,
                                 0, _lib.ptr(ws), ws.numel(), G.stream())
    assert rc == -4 and b"workspace" in lib.st2_last_error()
    torch.cuda.synchronize()


# ---------------------------------------------------------------- tensor-core paths
TC_SHAPES_T5 = {"encode": (5, 1024), "decode.3": (10, 512), "generator.noise_res.0.iter2": (100, 256),
                "generator.stage0.in": (100, 256), "generator.stage0.out": (100, 256),
                "generator.stage1.out": (500, 128), "generator.stage2.out": (1500, 64),
                "generator.noise_res.3.iter2": (3000, 32), "generator.stage3.out": (3000, 32)}


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
def test_hifigan_small_tensor_core_taps_and_snr(prec):
    """BASELINE.json north_star: 16-bit tensor-core path SNR >= 40 dB and per-layer relative L2 <= 1e-2."""
    cfg = DecoderConfig.hifigan()
    inp = np_inputs(2, 5, 1001, cfg)
    m = _decoder(cfg)
    out, ref, res = _tap_table(m, cfg, inp, TC_SHAPES_T5, precision=prec)
    for n, v in res.items():
        G.log("hifigan_small_tc_tap", prec=prec, tap=n, rel_l2=v)
    snr = snr_db(ref, out)
    G.log("hifigan_small_tc", prec=prec, snr_db=snr, maxabs=float(np.abs(out - ref).max()), launches=m.last_launch_count())
    for n, v in res.items():
        assert v <= 1e-2, (n, v)
    assert snr >= 40.0


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
def test_hifigan_cfg1_3s_tensor_core_snr(prec):
    cfg = DecoderConfig.hifigan()
    g = golden("hifigan_B1_T120_w0_i1001.npz")
    m = _decoder(cfg)
    out = _run(m, np_inputs(1, 120, 1001, cfg), precision=prec)
    snr = snr_db(g["out"], out)
    G.log("hifigan_cfg1_tc", prec=prec, snr_db=snr, maxabs=float(np.abs(out - g["out"]).max()))
    assert snr >= 40.0


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
def test_istftnet_small_tensor_core_snr(prec):
    cfg = DecoderConfig.istftnet()
    g = golden("istftnet_B2_T5_w0_i1005.npz")
    m = _decoder(cfg)
    out = _run(m, np_inputs(2, 5, 1005, cfg), precision=prec)
    snr = snr_db(g["out"], out)
    G.log("istftnet_small_tc", prec=prec, snr_db=snr, maxabs=float(np.abs(out - g["out"]).max()))
    assert snr >= 40.0


def test_fp16_intra_block_tensor_costs_little():
    """The fused resblocks keep six kinds of stage-private tensors in fp16 (DESIGN.md section 3: conv1 output, the running
    tensor between iterations, the stage input, the partial sum over the resblocks, the noise_convs output that feeds noise_res,
    the last stage's output that feeds conv_post); option "fp16_storage" / "fp16_xt" = 0 turns all of them off, "fp16_run" /
    "fp16_xu" / "fp16_sum" / "fp16_src" / "fp16_out" one kind each.
    Against the fp32-stored variant the waveform differs by about as much as two bf16 runs with different rounding do
    (bound 45 dB) and the SNR against the reference stays within a few tenths of a dB (bar 40 dB)."""
    cfg = DecoderConfig.hifigan()
    g = golden("hifigan_B1_T120_w0_i1001.npz")
    m = _decoder(cfg)
    lib = _lib.load()
    inp = np_inputs(1, 120, 1001, cfg)
    out16 = _run(m, inp, precision="bf16")
    # everything fp32: the module attribute (B200Decoder(..., fp16_storage=False) / st2_decoder_set_option)
    m.fp16_storage = False
    m.refresh_weights()
    try:
        out32 = _run(m, inp, precision="bf16")
    finally:
        m.fp16_storage = True
        m.refresh_weights()
    d = snr_db(out32, out16)
    G.log("xt16_vs_xt32", snr_between_db=d, snr16=snr_db(g["out"], out16), snr32=snr_db(g["out"], out32))
    assert not np.array_equal(out16, out32)      # the fp16 path really ran
    assert d >= 45.0
    assert snr_db(g["out"], out16) >= 40.0
    assert snr_db(g["out"], out16) >= snr_db(g["out"], out32) - 1.0
    assert np.array_equal(_run(m, inp, precision="bf16"), out16)
    assert lib.st2_decoder_set_option(m._handle, b"no_such_option", 1) == -1
    assert lib.st2_set_tuning(b"no_such_switch", 1) == -1
    # "fp16_xt" = 0 turns all four kinds off (the others build on the fp16 conv1 output) ...
    _lib.check(lib.st2_decoder_set_option(m._handle, b"fp16_xt", 0))
    try:
        assert np.array_equal(_run(m, inp, precision="bf16"), out32)
    finally:
        _lib.check(lib.st2_decoder_set_option(m._handle, b"fp16_xt", 1))
    # ... and each of the other five alone changes the result (the path it guards really runs) within the same bound
    for knob in (b"fp16_run", b"fp16_xu", b"fp16_sum", b"fp16_src", b"fp16_out"):
        _lib.check(lib.st2_decoder_set_option(m._handle, knob, 0))
        try:
            o = _run(m, inp, precision="bf16")
        finally:
            _lib.check(lib.st2_decoder_set_option(m._handle, knob, 1))
        assert not np.array_equal(o, out16), knob
        assert snr_db(out32, o) >= 45.0 and snr_db(g["out"], o) >= 40.0, knob
    assert np.array_equal(_run(m, inp, precision="bf16"), out16)


@pytest.mark.parametrize("variant,B,T", [("hifigan", 8, 400), ("istftnet", 1, 2400), ("hifigan", 3, 203)])
def test_full_size_tensor_core_path_tracks_fp32_path(variant, B, T):
    """BASELINE.json configs[3] / [4] sizes (10 s utterances; the 60 s iSTFTNet long form) and a ragged length: the oracle
    is too slow there, so the bf16 tensor-core path (TMA pipeline kernels, multi-hundred-tile persistent loops, ragged last
    tiles) is checked against the fp32 SIMT path of the same library, which the small-size tests pin to the reference.
    Bar: SNR >= 40 dB, finite output of the right shape."""
    cfg = DecoderConfig.hifigan() if variant == "hifigan" else DecoderConfig.istftnet()
    m = _decoder(cfg)
    inp = synth.make_inputs(B, T, seed=2000 + T, cfg=cfg, with_noise=False)
    t = {k: v.cuda() for k, v in inp.items()}
    with torch.no_grad():
        ref = m(t["asr"], t["F0_curve"], t["N"], t["s"], seed=77, precision="fp32").float().cpu().numpy()
        out = m(t["asr"], t["F0_curve"], t["N"], t["s"], seed=77, precision="bf16").float().cpu().numpy()
    assert out.shape == (B, 1, 600 * T) and np.isfinite(out).all()
    snr = snr_db(ref, out)
    G.log("full_size_tc_vs_fp32", variant=variant, B=B, T=T, snr_db=snr)
    assert snr >= 40.0


def test_conv_row_inline_coefficients_match_the_coefficient_kernel():
    """At sizes where the 32 / 64-channel resblocks run on conv_row.cu a launch fed by another conv_row launch computes its AdaIN
    coefficients itself (39 fewer launches per forward).  Same partials, same fp64 arithmetic, another summation order than
    adain_coef_row_kernel: against the build with the switch off the waveform must agree to rounding noise (>= 80 dB), the
    launch count must really drop, and the path must be bit-reproducible."""
    cfg = DecoderConfig.hifigan()
    m = _decoder(cfg)
    lib = _lib.load()
    inp = synth.make_inputs(8, 400, seed=2400, cfg=cfg, with_noise=False)
    t = {k: v.cuda() for k, v in inp.items()}

    def run():
        with torch.no_grad():
            o = m(t["asr"], t["F0_curve"], t["N"], t["s"], seed=78, precision="bf16").float().cpu().numpy()
        return o, m.last_launch_count()
    a, na = run()
    a2, _ = run()
    _lib.check(lib.st2_set_tuning(b"no_row_inline_coef", 1))
    try:
        b, nb = run()
    finally:
        _lib.check(lib.st2_set_tuning(b"no_row_inline_coef", 0))
    assert np.array_equal(a, a2)
    assert nb - na >= 30, (na, nb)
    assert snr_db(b, a) >= 80.0, snr_db(b, a)


@pytest.mark.parametrize("variant", ["hifigan", "istftnet"])
def test_cuda_graph_replay_matches_eager(variant):
    """forward(..., cuda_graph=True) captures the launches once per shape and replays them; the Philox seed is read from
    device memory, so a replay with another seed must equal the eager forward with that seed bit for bit."""
    cfg = DecoderConfig.hifigan() if variant == "hifigan" else DecoderConfig.istftnet()
    m = _decoder(cfg)
    for B, T in ((1, 30), (2, 12)):
        a = {k: v.cuda() for k, v in synth.make_inputs(B, T, seed=50 + T, cfg=cfg, with_noise=False).items()}
        b = {k: v.cuda() for k, v in synth.make_inputs(B, T, seed=60 + T, cfg=cfg, with_noise=False).items()}
        with torch.no_grad():
            for inp, seed in ((a, 11), (b, 2 ** 63 + 5), (a, 12)):
                eager = m(inp["asr"], inp["F0_curve"], inp["N"], inp["s"], seed=seed, precision="bf16")
                graph = m(inp["asr"], inp["F0_curve"], inp["N"], inp["s"], seed=seed, precision="bf16", cuda_graph=True)
                torch.cuda.synchronize()
                assert torch.equal(eager, graph), (variant, B, T, seed)
            e1 = m(a["asr"], a["F0_curve"], a["N"], a["s"], seed=11, precision="bf16")
            e2 = m(a["asr"], a["F0_curve"], a["N"], a["s"], seed=12, precision="bf16")
            assert not torch.equal(e1, e2)       # the seed really changes the noise


def test_pipelined_serving_loop_matches_direct_forward():
    """streaming.PipelinedDecoder (pinned H2D / forward / pinned D2H on three streams) returns, batch by batch and in order,
    exactly what the module returns for the same inputs and seeds -- including a change of shape between batches."""
    from styletts2_lite_b200.streaming import PipelinedDecoder
    cfg = DecoderConfig.hifigan()
    m = _decoder(cfg)
    shapes = [(2, 9), (2, 9), (3, 14), (2, 9), (1, 30)]
    batches = [{k: v.pin_memory() for k, v in synth.make_inputs(B, T, seed=300 + i, cfg=cfg, with_noise=False).items()}
               for i, (B, T) in enumerate(shapes)]
    direct = []
    with torch.no_grad():
        for i, b in enumerate(batches):
            direct.append(m(b["asr"].cuda(), b["F0_curve"].cuda(), b["N"].cuda(), b["s"].cuda(), seed=900 + i,
                            precision="bf16").cpu())
    pipe = PipelinedDecoder(m, precision="bf16")
    got = [w.clone() for w in pipe.decode(batches, iter(range(900, 900 + len(batches))))]
    assert len(got) == len(direct)
    for i, (a, b) in enumerate(zip(direct, got)):
        assert a.shape == b.shape and torch.equal(a, b), i
    assert list(pipe.decode([])) == []


# ---------------------------------------------------------------- round-2 fixtures: longer / ragged / true-init cases
@pytest.mark.parametrize("name,variant,T,ws,iseed,perturb", [
    ("hifigan_B1_T120_w3_i1007_plain", "hifigan", 120, 3, 1007, False),
    ("hifigan_B1_T203_w0_i1009", "hifigan", 203, 0, 1009, True),
    ("istftnet_B1_T120_w0_i1006", "istftnet", 120, 0, 1006, True),
    ("istftnet_B1_T203_w0_i1008", "istftnet", 203, 0, 1008, True),
    ("hifigan_B1_T400_w0_i1003", "hifigan", 400, 0, 1003, True)])
def test_fp32_path_vs_reference_goldens_long_and_ragged(name, variant, T, ws, iseed, perturb):
    """fp32 path max-abs <= 1e-4 against waveforms of the unmodified reference (tests/golden/make_golden_r2.py): 3 s with the
    reference's true initialisation, ragged lengths no tile size divides, 3 s iSTFTNet and the 10 s case where SineGen phases
    reach 1e5 rad (SURVEY.md: the hardest case for fp32 parity)."""
    cfg = DecoderConfig.hifigan() if variant == "hifigan" else DecoderConfig.istftnet()
    g = golden(name + ".npz")
    m = _decoder(cfg, ws, perturb)
    out = _run(m, np_inputs(1, T, iseed, cfg))
    err = float(np.abs(out - g["out"]).max())
    G.log("fp32_vs_reference_golden", fixture=name, maxabs=err, snr_db=snr_db(g["out"], out))
    assert out.shape == g["out"].shape
    assert err <= 1e-4


@pytest.mark.parametrize("name,variant,T,ws,iseed,perturb", [
    ("hifigan_B1_T120_w3_i1007_plain", "hifigan", 120, 3, 1007, False),
    ("hifigan_B1_T203_w0_i1009", "hifigan", 203, 0, 1009, True),
    ("istftnet_B1_T120_w0_i1006", "istftnet", 120, 0, 1006, True),
    ("istftnet_B1_T203_w0_i1008", "istftnet", 203, 0, 1008, True),
    ("hifigan_B1_T400_w0_i1003", "hifigan", 400, 0, 1003, True)])
@pytest.mark.parametrize("prec", ["bf16", "fp16"])
def test_tensor_core_paths_vs_reference_goldens_long_and_ragged(name, variant, T, ws, iseed, perturb, prec):
    """16-bit paths (fp16 stage-private tensors on, the default) against the same reference waveforms: SNR >= 40 dB -- on the
    reference's true initialisation too, and at 10 s."""
    cfg = DecoderConfig.hifigan() if variant == "hifigan" else DecoderConfig.istftnet()
    g = golden(name + ".npz")
    m = _decoder(cfg, ws, perturb)
    out = _run(m, np_inputs(1, T, iseed, cfg), precision=prec)
    snr = snr_db(g["out"], out)
    G.log("tc_vs_reference_golden", fixture=name, prec=prec, snr_db=snr, maxabs=float(np.abs(out - g["out"]).max()))
    assert snr >= 40.0


def test_bf16_every_resblock_tap_at_3s():
    """BASELINE.json: per-layer relative L2 <= 1e-2 on the bf16 path.  Every conv1 output (`.convs1.j`), every running tensor
    (`.iterj`) and every stage input / output of the generator at T = 120 (3 s: tensors of up to 72,000 rows, hundreds of
    tiles, the fp16-stored ones included) against the taps of the torch CPU port of the reference (oracle/decoder_torch.py,
    pinned bit-tight to the reference goldens by tests/test_oracle.py)."""
    from oracle import decoder_torch as OT
    cfg = DecoderConfig.hifigan()
    T = 120
    m = _decoder(cfg)
    inp = np_inputs(1, T, 1001, cfg)
    names = {"encode": (T, 1024), "decode.0": (T, 1024), "decode.3": (2 * T, 512)}
    lens = [20 * T, 100 * T, 300 * T, 600 * T]
    for i in range(4):
        C_ = 256 >> i
        names["generator.stage%d.in" % i] = (lens[i], C_)
        names["generator.stage%d.out" % i] = (lens[i], C_)
        for blk in ["generator.noise_res.%d" % i] + ["generator.resblocks.%d" % (3 * i + j) for j in range(3)]:
            for j in range(3):
                names["%s.convs1.%d" % (blk, j)] = (lens[i], C_)
                if j < 2 or "noise_res" in blk:
                    names["%s.iter%d" % (blk, j)] = (lens[i], C_)
    bufs = {n: m.set_tap(n, 1, rows, C_) for n, (rows, C_) in names.items()}
    out = _run(m, inp, precision="bf16")
    taps = {}
    W = OT.TorchWeights(synth.make_state_dict(cfg, 0, True))
    ti = {k: torch.from_numpy(v) for k, v in inp.items()}
    ref = OT.decoder_forward(W, cfg, ti["asr"], ti["F0_curve"], ti["N"], ti["s"], ti["noise"], taps=taps).numpy()
    worst = ("", 0.0)
    for n, buf in bufs.items():
        v = rel_l2(taps[n].numpy(), G.cf(buf.cpu().numpy()))
        if v > worst[1]:
            worst = (n, v)
        if v > 5e-3:
            G.log("bf16_tap_T120", tap=n, rel_l2=v)
        assert v <= 1e-2, (n, v)
    m.clear_taps()
    snr = snr_db(ref, out)
    G.log("bf16_every_tap_T120", taps=len(bufs), worst_tap=worst[0], worst_rel_l2=worst[1], snr_db=snr)
    assert snr >= 40.0


def test_bench_shape_bf16_tracks_fp32():
    """The shape bench.py times (BASELINE.json configs[1]: 64 x 5 s): bf16 path against the fp32 path of this library,
    SNR >= 40 dB, every utterance finite and individually >= 38 dB."""
    cfg = DecoderConfig.hifigan()
    m = _decoder(cfg)
    B, T = 64, 200
    inp = synth.make_inputs(B, T, seed=1002, cfg=cfg, with_noise=False)
    t = {k: v.cuda() for k, v in inp.items()}
    with torch.no_grad():
        ref = m(t["asr"], t["F0_curve"], t["N"], t["s"], seed=5, precision="fp32").float().cpu().numpy()
        out = m(t["asr"], t["F0_curve"], t["N"], t["s"], seed=5, precision="bf16").float().cpu().numpy()
    assert out.shape == (B, 1, 600 * T) and np.isfinite(out).all()
    snr = snr_db(ref, out)
    per = [snr_db(ref[b], out[b]) for b in range(B)]
    G.log("bench_shape_bf16_vs_fp32", snr_db=snr, worst_utterance_db=min(per))
    assert snr >= 40.0 and min(per) >= 38.0


def test_graph_cache_is_bounded_and_profiling_falls_back_to_eager():
    """ADVICE r1: (1) the CUDA-graph cache is an LRU with a bound (each entry owns a workspace); (2) with the per-launch event
    profile on, cuda_graph=True runs eagerly (events recorded during capture would be garbage) and the profile stays sane."""
    cfg = DecoderConfig.hifigan()
    m = _decoder(cfg)
    old = m.max_graphs
    m.max_graphs = 2
    try:
        m._graphs.clear()
        ins = {T: {k: v.cuda() for k, v in synth.make_inputs(1, T, seed=70 + T, cfg=cfg, with_noise=False).items()} for T in (6, 7, 8)}
        with torch.no_grad():
            for T in (6, 7, 8, 6):
                a = ins[T]
                e = m(a["asr"], a["F0_curve"], a["N"], a["s"], seed=9, precision="bf16")
                g = m(a["asr"], a["F0_curve"], a["N"], a["s"], seed=9, precision="bf16", cuda_graph=True)
                assert torch.equal(e, g), T
                assert len(m._graphs) <= 2
        assert [k[1] for k in m._graphs] == [8, 6]              # 7 was the least recently used shape when 6 came back
        m.set_profiling(True)
        with torch.no_grad():
            a = ins[6]
            g = m(a["asr"], a["F0_curve"], a["N"], a["s"], seed=9, precision="bf16", cuda_graph=True)
        prof = m.get_profile()
        m.set_profiling(False)
        assert torch.equal(g, e)
        total = sum(v["ms"] for v in prof.values())
        n_prof = sum(v["launches"] for v in prof.values())          # a few setup launches share one profile record
        assert 0.05 < total < 200.0 and m.last_launch_count() - 8 <= n_prof <= m.last_launch_count()
    finally:
        m.set_profiling(False)
        m.max_graphs = old


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs in one process")
def test_two_devices_in_one_process():
    """ADVICE r1 (medium): one-time function attributes (> 48 KB dynamic shared memory) and the SM count are cached per device,
    so a second GPU driven from the same process launches the large-shared-memory kernels too and agrees bit for bit."""
    cfg = DecoderConfig.hifigan()
    sd = synth.make_state_dict(cfg, 0, True)
    inp = synth.make_inputs(2, 40, seed=31, cfg=cfg, with_noise=False)
    outs = []
    for d in (0, 1):
        m = B200Decoder(cfg, "bf16")
        m.load_state_dict(sd)
        m = m.to("cuda:%d" % d).eval()
        t = {k: v.to("cuda:%d" % d) for k, v in inp.items()}
        with torch.no_grad():
            outs.append(m(t["asr"], t["F0_curve"], t["N"], t["s"], seed=3).cpu())
        torch.cuda.synchronize(d)
    assert torch.isfinite(outs[0]).all() and torch.equal(outs[0], outs[1])


def test_torch_port_on_the_gpu_matches_golden():
    """bench.py's eager_gpu leg runs oracle/decoder_torch.py on the GPU when the unmodified reference modules are not staged:
    on CUDA tensors (TF32 off) it reproduces the reference waveforms it is pinned to on the host."""
    from oracle import decoder_torch as OT
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        for cfg, name, seed in ((DecoderConfig.hifigan(), "hifigan_B2_T5_w0_i1001.npz", 1001),
                                (DecoderConfig.istftnet(), "istftnet_B2_T5_w0_i1005.npz", 1005)):
            W = OT.TorchWeights({k: v.cuda() for k, v in synth.make_state_dict(cfg, 0, True).items()})
            t = {k: v.cuda() for k, v in synth.make_inputs(2, 5, seed, cfg).items()}
            out = OT.decoder_forward(W, cfg, t["asr"], t["F0_curve"], t["N"], t["s"], t["noise"]).cpu().numpy()
            err = float(np.abs(out - golden(name)["out"]).max())
            G.log("torch_port_gpu_vs_golden", fixture=name, maxabs=err)
            assert err <= 1e-3, (name, err)
    finally:
        torch.backends.cudnn.allow_tf32 = tf32


# ---------------------------------------------------------------- §8(f) N4: the Vocos decoder variant (Modules/vocos.py)
def _vocos_inputs(B, T, seed, cfg):
    return {k: v.numpy() for k, v in synth.make_inputs(B, T, seed, cfg, with_noise=False).items()}


def _run_vocos(m, inp, precision="fp32"):
    t = {k: torch.from_numpy(v).cuda() for k, v in inp.items()}
    with torch.no_grad():
        out = m(t["asr"], t["F0_curve"], t["N"], t["s"], precision=precision)
    torch.cuda.synchronize()
    return out.cpu().numpy()


def test_vocos_small_fp32_golden_and_taps():
    """Reference fixture of the unmodified Modules/vocos.py Decoder (tests/golden/make_golden_vocos.py): waveform <= 1e-4 and
    the taps of the front half, the first / last ConvNeXt block, the final LayerNorm and ISTFTHead.out."""
    cfg = DecoderConfig.vocos()
    g = golden("vocos_B2_T6_w0_i1000.npz")
    m = _decoder(cfg)
    T = 6
    shapes = {"decode.3": (2 * T, 512), "generator.convnext.0.dwconv": (2 * T, 512), "generator.convnext.0": (2 * T, 512),
              "generator.convnext.7": (2 * T, 512), "generator.final_layer_norm": (2 * T, 512), "generator.stft.out": (2 * T, 1202)}
    bufs = {n: m.set_tap(n, 2, rows, C_) for n, (rows, C_) in shapes.items()}
    out = _run_vocos(m, _vocos_inputs(2, T, 1000, cfg))
    m.clear_taps()
    assert out.shape == (2, 1, 3600)
    assert np.abs(G.cf(bufs["decode.3"].cpu().numpy()) - g["tap:decode.3"]).max() <= 1e-4
    for n in ("generator.convnext.0", "generator.convnext.7"):
        assert np.abs(G.cf(bufs[n].cpu().numpy()) - g["tap:" + n]).max() <= 1e-4, n
    assert np.abs(bufs["generator.final_layer_norm"].cpu().numpy() - g["tap:generator.final_layer_norm"]).max() <= 1e-4
    assert np.abs(bufs["generator.stft.out"].cpu().numpy() - g["tap:generator.stft.out"]).max() <= 1e-4
    assert np.abs(out - g["out"]).max() <= 1e-4
    # the oracle's depthwise conv (no reference hook sits between dwconv and norm)
    taps = {}
    sd = {k: v.numpy() for k, v in synth.make_state_dict(cfg, 0, True).items()}
    inp = _vocos_inputs(2, T, 1000, cfg)
    O.decoder_forward(sd, cfg, inp["asr"], inp["F0_curve"], inp["N"], inp["s"], None, taps=taps)
    assert np.abs(G.cf(bufs["generator.convnext.0.dwconv"].cpu().numpy()) - taps["generator.convnext.0.dwconv"]).max() <= 2e-5


def test_vocos_3s_fp32_golden_and_tensor_core_paths():
    cfg = DecoderConfig.vocos()
    g = golden("vocos_B1_T120_w0_i1001.npz")
    m = _decoder(cfg)
    inp = _vocos_inputs(1, 120, 1001, cfg)
    out = _run_vocos(m, inp)
    assert out.shape == (1, 1, 72000) and np.abs(out - g["out"]).max() <= 1e-4
    for prec in ("bf16", "fp16"):
        o16 = _run_vocos(m, inp, prec)
        assert snr_db(g["out"], o16) >= 40.0, (prec, snr_db(g["out"], o16))


def test_vocos_batch_sizes_and_independence_vs_oracle():
    """Odd frame counts (tiles that are not full), T = 3 (6 frames: barely longer than the 4-frame ISTFT overlap; at T = 2 the
    front half's InstanceNorm over two samples amplifies fp32 rounding beyond any tolerance, on the CPU as well), a batch with
    different styles: each utterance equals its own B = 1 call bit for bit, and the oracle on two of them."""
    cfg = DecoderConfig.vocos()
    m = _decoder(cfg)
    sd = {k: v.numpy() for k, v in synth.make_state_dict(cfg, 0, True).items()}
    for B, T, seed in ((3, 37, 1010), (2, 3, 1011), (5, 203, 1012)):
        inp = _vocos_inputs(B, T, seed, cfg)
        out = _run_vocos(m, inp)
        assert out.shape == (B, 1, 600 * T) and np.isfinite(out).all()
        one = _run_vocos(m, {k: v[B - 1:B] for k, v in inp.items()})
        assert np.array_equal(out[B - 1:B], one)
        nb = 1 if T > 100 else 2
        ref = O.decoder_forward(sd, cfg, inp["asr"][:nb], inp["F0_curve"][:nb], inp["N"][:nb], inp["s"][:nb], None)
        assert np.abs(out[:nb] - ref).max() <= 1e-4, (B, T)


def test_vocos_drop_in_constructor_and_graph_replay():
    from styletts2_lite_b200 import vocos
    m = vocos.Decoder(dim_in=512, style_dim=128, dim_out=80, intermediate_dim=1536, num_layers=8, gen_istft_n_fft=1200,
                      gen_istft_hop_size=300, precision="bf16")
    assert sum(p.numel() for p in m.parameters()) == 47_919_258 and len(m.state_dict()) == 149
    cfg = DecoderConfig.vocos()
    m.load_state_dict(synth.make_state_dict(cfg, 0, True))
    m = m.to("cuda").eval()
    inp = {k: v.cuda() for k, v in synth.make_inputs(2, 40, 1013, cfg, with_noise=False).items()}
    with torch.no_grad():
        a = m(inp["asr"], inp["F0_curve"], inp["N"], inp["s"])
        b = m(inp["asr"], inp["F0_curve"], inp["N"], inp["s"], cuda_graph=True)
        c = m(inp["asr"], inp["F0_curve"], inp["N"], inp["s"], cuda_graph=True)
    assert torch.equal(a, b) and torch.equal(b, c)
    ref = _run_vocos(_decoder(cfg), {k: v.cpu().numpy() for k, v in inp.items()})
    assert snr_db(ref, a.cpu().numpy()) >= 40.0


def test_vocos_other_head_geometry_vs_oracle():
    """The reference constructor's own defaults for the ISTFT head (n_fft 1024, hop 256: Modules/vocos.py:366-368) with a smaller
    backbone (2 blocks, intermediate 1024): 512 samples per asr frame, operand padding 1026 -> 1152, 4 frames per sample again."""
    from styletts2_lite_b200 import vocos
    m = vocos.Decoder(dim_in=512, style_dim=128, dim_out=80, intermediate_dim=1024, num_layers=2, gen_istft_n_fft=1024,
                      gen_istft_hop_size=256)
    cfg = m.cfg
    assert cfg.samples_per_frame == 512
    sdt = synth.make_state_dict(cfg, 3, True)
    m.load_state_dict(sdt)
    m = m.to("cuda").eval()
    inp = synth.make_inputs(2, 9, 1020, cfg, with_noise=False)
    with torch.no_grad():
        out = m(inp["asr"].cuda(), inp["F0_curve"].cuda(), inp["N"].cuda(), inp["s"].cuda()).cpu().numpy()
        o16 = m(inp["asr"].cuda(), inp["F0_curve"].cuda(), inp["N"].cuda(), inp["s"].cuda(), precision="fp16").cpu().numpy()
    ref = O.decoder_forward({k: v.numpy() for k, v in sdt.items()}, cfg, inp["asr"].numpy(), inp["F0_curve"].numpy(),
                            inp["N"].numpy(), inp["s"].numpy(), None)
    assert out.shape == ref.shape == (2, 1, 512 * 9)
    assert np.abs(out - ref).max() <= 1e-4
    assert snr_db(ref, o16) >= 40.0
