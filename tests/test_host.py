"""CPU tests (-m "not gpu"): the C-ABI library loads and exports every symbol include/st2_b200.h
declares (no compute calls), the drop-in module mirrors the reference's state_dict schema, and the
host logic fails loudly without a GPU."""
import json
import os
import re

import pytest
import torch

from styletts2_lite_b200 import _lib, synth
from styletts2_lite_b200.config import DecoderConfig, buffer_specs, param_specs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from styletts2_lite_b200 import build
    build.build()                                  # nvcc cross-compiles sm_100a without a GPU
    return _lib.load()


def _header_functions():
    src = open(os.path.join(ROOT, "include", "st2_b200.h")).read()
    return re.findall(r"^ST2_API\s+[\w\s\*]+?\b(st2_\w+)\(", src, flags=re.M)


def test_library_exports_every_declared_symbol(lib):
    names = _header_functions()
    assert len(names) >= 19
    for n in names:
        assert hasattr(lib, n), n
    assert sorted(names) == sorted(_lib.SIGNATURES)
    assert lib.st2_abi_version() == 1


def test_create_validates_config_without_gpu(lib):
    import ctypes as C
    cc = _lib.St2Config.from_config(DecoderConfig.hifigan())
    cc.variant = 7
    h = C.c_void_p()
    assert lib.st2_decoder_create(C.byref(cc), C.byref(h)) == -1
    assert b"variant" in lib.st2_last_error()
    cc = _lib.St2Config.from_config(DecoderConfig.istftnet())
    assert lib.st2_decoder_create(C.byref(cc), C.byref(h)) == 0
    assert lib.st2_decoder_workspace_bytes(h, 1, 10, 0) == -2        # not finalized
    lib.st2_decoder_destroy(h)
    cc = _lib.St2Config.from_config(DecoderConfig.vocos())               # the third decoder.type (Modules/vocos.py)
    assert cc.variant == 4 and cc.num_layers == 8 and cc.intermediate_dim == 1536
    assert lib.st2_decoder_create(C.byref(cc), C.byref(h)) == 0
    lib.st2_decoder_destroy(h)
    cc.gen_istft_hop_size = 301                                          # n_fft - hop must be even ('same' padding, vocos.py:203)
    assert lib.st2_decoder_create(C.byref(cc), C.byref(h)) == -1


def test_set_tuning_accepts_only_the_test_hooks(lib):
    for name in (b"no_pipe", b"row_always", b"row_sub", b"no_row_inline_coef", b"verbose"):
        assert lib.st2_set_tuning(name, 0) == 0, name          # 0 is each hook's default: no state changes
    for name in (b"pipe_xmax", b"no_row", b"tc_halo", b"no_xt16", b"lstm_bt"):
        assert lib.st2_set_tuning(name, 0) == -1, name
        assert b"unknown switch" in lib.st2_last_error()


@pytest.mark.parametrize("variant", ["hifigan", "istftnet", "vocos"])
def test_state_dict_schema_matches_reference(variant):
    schema = json.load(open(os.path.join(ROOT, "tests", "golden", "state_dict_schema.json")))[variant]
    cfg = {"hifigan": DecoderConfig.hifigan, "istftnet": DecoderConfig.istftnet, "vocos": DecoderConfig.vocos}[variant]()
    mine = {n: list(s) for n, s, _ in param_specs(cfg)}
    mine.update({n: list(s) for n, s in buffer_specs(cfg)})
    assert mine == schema["state_dict"]
    from styletts2_lite_b200.decoder import B200Decoder
    m = B200Decoder(cfg)
    assert {k: list(v.shape) for k, v in m.state_dict().items()} == schema["state_dict"]
    assert sum(p.numel() for p in m.parameters()) == schema["num_params"]
    sd = synth.make_state_dict(cfg, 0, True)
    r = m.load_state_dict(sd)
    assert not r.missing_keys and not r.unexpected_keys
    # the reference's fallback strips a 7-char 'module.' prefix (inference.py:165-168): plain keys must load
    key = "generator.stft.out.weight" if variant == "vocos" else "generator.conv_post.weight_v"
    assert torch.equal(m.state_dict()[key], sd[key])
    if variant == "vocos":
        from styletts2_lite_b200.vocos import Decoder
        m2 = Decoder(dim_in=512, style_dim=128, dim_out=80, intermediate_dim=1536, num_layers=8, gen_istft_n_fft=1200,
                     gen_istft_hop_size=300)                             # models.py:555-562
        assert set(m2.state_dict()) == set(schema["state_dict"]) and m2.cfg.samples_per_frame == 600


def test_predictor_state_dict_schema_matches_reference():
    """F0Ntrain subset of ProsodyPredictor.state_dict() (models.py:407-419), checked against the reference module when
    the fixture was made; a full predictor state_dict loads with the duration half ignored."""
    from styletts2_lite_b200.config import PredictorConfig, predictor_param_specs
    from styletts2_lite_b200.predictor import B200F0NPredictor
    schema = json.load(open(os.path.join(ROOT, "tests", "golden", "state_dict_schema.json")))["predictor_f0n"]
    assert {n: list(s) for n, s, _ in predictor_param_specs(PredictorConfig())} == schema["state_dict"]
    m = B200F0NPredictor(style_dim=128, d_hid=512, nlayers=3, max_dur=50, dropout=0.2)
    assert {k: list(v.shape) for k, v in m.state_dict().items()} == schema["state_dict"]
    sd = synth.make_predictor_state_dict(seed=0)
    full = dict(sd)
    full["duration_proj.linear_layer.weight"] = torch.zeros(50, 512)      # entries of the duration half are skipped
    full["lstm.weight_ih_l0"] = torch.zeros(1024, 640)
    r = m.load_state_dict(full)
    assert not r.missing_keys and not r.unexpected_keys
    assert torch.equal(m.state_dict()["shared.weight_hh_l0_reverse"], sd["shared.weight_hh_l0_reverse"])
    with pytest.raises(Exception):
        m.F0Ntrain(torch.zeros(1, 640, 4), torch.zeros(1, 128))           # no CPU path
    # with duration=True the module holds every parameter of the reference ProsodyPredictor
    from styletts2_lite_b200.config import duration_param_specs
    full = json.load(open(os.path.join(ROOT, "tests", "golden", "state_dict_schema.json")))["predictor"]
    m2 = B200F0NPredictor(style_dim=128, d_hid=512, nlayers=3, max_dur=50, dropout=0.2, duration=True)
    assert {k: list(v.shape) for k, v in m2.state_dict().items()} == full["state_dict"]
    assert sum(p.numel() for p in m2.parameters()) == full["num_params"]
    r = m2.load_state_dict(synth.make_predictor_state_dict(seed=0, duration=True))
    assert not r.missing_keys and not r.unexpected_keys


def test_text_encoder_state_dict_schema_matches_reference():
    from styletts2_lite_b200.text_encoder import B200TextEncoder
    schema = json.load(open(os.path.join(ROOT, "tests", "golden", "state_dict_schema.json")))["text_encoder"]
    m = B200TextEncoder(channels=512, kernel_size=5, depth=3, n_symbols=178)
    assert {k: list(v.shape) for k, v in m.state_dict().items()} == schema["state_dict"]
    assert sum(p.numel() for p in m.parameters()) == schema["num_params"]
    r = m.load_state_dict(synth.make_text_state_dict(seed=0))
    assert not r.missing_keys and not r.unexpected_keys
    with pytest.raises(Exception):
        m(torch.zeros(1, 4, dtype=torch.long))                            # no CPU path


def test_no_cpu_fallback():
    from styletts2_lite_b200 import hifigan, length_regulator
    m = hifigan.Decoder(style_dim=128)
    with pytest.raises(_lib.St2Error):
        m(torch.zeros(1, 512, 4), torch.zeros(1, 8), torch.zeros(1, 8), torch.zeros(1, 128))
    m.train(True)
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 512, 4), torch.zeros(1, 8), torch.zeros(1, 8), torch.zeros(1, 128))
    with pytest.raises(_lib.St2Error):
        length_regulator.round_durations(torch.ones(1, 4))


def test_product_package_does_not_import_oracle():
    pkg = os.path.join(ROOT, "styletts2_lite_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f
                assert "decoder_np" not in src and "oracle/" not in src, f


def test_synth_is_deterministic():
    cfg = DecoderConfig.hifigan()
    a, b = synth.make_inputs(2, 6, 5, cfg), synth.make_inputs(2, 6, 5, cfg)
    assert all(torch.equal(a[k], b[k]) for k in a)
    assert (a["F0_curve"] == 0).float().mean() > 0.1
    d = synth.make_durations(4, 64, 320)
    assert d.shape == (4, 64) and (d >= 1).all() and (d.sum(1) == 320).all()
