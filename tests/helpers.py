"""Shared helpers for the test-suite (CPU + GPU)."""
import hashlib
import os

import numpy as np

from styletts2_lite_b200.config import DecoderConfig
from styletts2_lite_b200 import synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def np_state_dict(cfg, seed=0, perturb=True):
    return {k: v.numpy() for k, v in synth.make_state_dict(cfg, seed, perturb).items()}


def np_inputs(B, T, seed, cfg=None, with_noise=True):
    return {k: v.numpy() for k, v in synth.make_inputs(B, T, seed, cfg, with_noise).items()}


def golden(name):
    return np.load(os.path.join(GOLDEN, name))


def resblock_tap_shapes(T, stages=range(4)):
    """{tap name: (rows, C)} of the HiFi-GAN generator's AdaINResBlock1 layers in `stages`: every conv1 output (`.convs1.j`),
    every running tensor (`.iterj`; the last one of a resblock is folded into the stage sum) and every stage input / output,
    for an utterance of T asr frames.  The names are the taps of oracle/decoder_torch.py and of B200Decoder.set_tap."""
    lens = [20 * T, 100 * T, 300 * T, 600 * T]
    names = {}
    for i in stages:
        C_ = 256 >> i
        names["generator.stage%d.in" % i] = (lens[i], C_)
        names["generator.stage%d.out" % i] = (lens[i], C_)
        for blk in ["generator.noise_res.%d" % i] + ["generator.resblocks.%d" % (3 * i + j) for j in range(3)]:
            for j in range(3):
                names["%s.convs1.%d" % (blk, j)] = (lens[i], C_)
                if j < 2 or "noise_res" in blk:
                    names["%s.iter%d" % (blk, j)] = (lens[i], C_)
    return names


def snr_db(ref, x):
    ref = ref.astype(np.float64)
    err = x.astype(np.float64) - ref
    return 10.0 * np.log10((ref ** 2).sum() / max((err ** 2).sum(), 1e-300))


def rel_l2(ref, x):
    ref = ref.astype(np.float64)
    return float(np.linalg.norm(x.astype(np.float64) - ref) / max(np.linalg.norm(ref), 1e-300))
