#!/usr/bin/env python
"""Benchmark of the decoder hot path (BASELINE.json metric: decoder audio-seconds per second).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

One "step" = Decoder.forward over one synthetic batch of BASELINE.json configs[1]
(hifigan, B=64 utterances x 5 s = T 200 frames, random-init weights, bf16 tensor-core path).
Rank 0 prints ONE JSON line.  For N>1 (torchrun) every rank runs its own batch (utterances
shard with no cross-rank math, weak scaling) and the waveforms are gathered to rank 0 over NCCL
inside the timed region: each step's batch goes point-to-point into its slice of one preallocated
buffer on rank 0, on a side stream, so the gather of step k overlaps the forward of step k+1
(parallel.ShardedGather).  Auxiliary keys (outside the timed region): `cfg4_sharded_1024x10s`
(N>1: BASELINE configs[3], 1024 x 10 s sharded in micro-batches, gathered to rank 0),
`cfg5_istftnet_60s` (configs[4]), `full_path_cfg3` (configs[2]) and `eager_gpu` (the reference
decoder through PyTorch eager on the same GPU, fp32 and bf16 autocast: the pre-existing GPU path).

  value     whole-job audio-s/s with inputs resident in HBM (CUDA events, max over ranks)
  e2e       same metric through the package's host-fed serving loop (streaming.PipelinedDecoder around the drop-in
            module): HOST (pinned) inputs copied in and the waveform copied back to pinned host memory every step,
            inside the timed region, overlapped with the neighbouring forwards on copy streams
  roofline  the dominant kernel (conv_row_kernel / conv_pipe_kernel: fused AdaIN/Snake -> tcgen05 conv -> residual/stats):
            algorithmic bytes / event-timed duration vs the measured HBM copy peak of MEASURED_PEAKS.json; `kernels` lists
            every kernel category with its time share, TFLOP/s and GB/s
  cpu_baseline  the reference decoder on the host cores (rank 0, N=1): the UNMODIFIED reference modules when they are staged
            under baseline/_ref (oracle/stage_reference.py; kind "reference"), else the torch-CPU port (kind "port")

--impl reference times that same CPU arm on a bounded sample of the workload (8 utterances per step).

--dump-outputs DIR writes the waveforms of the last timed step (gathered on rank 0 for N>1) as DIR/waveform.npy, float32
[utterances, 1, samples], so that two builds run with the same arguments (hence the same inputs, weights and noise seeds)
can be compared output for output.  Above 64 MiB it keeps a fixed, seeded sample of the utterances.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "decoder audio-sec/sec (RTF^-1)"
UNIT = "audio-s/s"
SR = 24000


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="utterances per GPU")
    ap.add_argument("--frames", type=int, default=200, help="asr frames per utterance (200 = 5 s)")
    ap.add_argument("--variant", default="hifigan", choices=["hifigan", "istftnet"])
    ap.add_argument("--precision", default="bf16", choices=["fp32", "bf16", "fp16"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-chain", action="store_true", help="skip the auxiliary BASELINE configs[2] measurement (full_path_cfg3)")
    ap.add_argument("--cpu-frames", type=int, default=0, help="frames of the CPU sample (default: --frames)")
    ap.add_argument("--cpu-batch", type=int, default=8, help="utterances per step of the CPU arm")
    ap.add_argument("--gather", default="p2p", choices=["direct", "p2p"],
                    help="N > 1: NCCL send / recv on a side stream (default), or decode straight into rank 0's buffer over NVLink "
                         "(symmetric memory; bit-identical, measured 1-2 %% slower per step at N = 2: the last kernel's stores go remote)")
    ap.add_argument("--no-aux", action="store_true", help="skip every auxiliary measurement (cfg3/cfg4/cfg5/eager_gpu)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the waveforms of the last timed step to DIR/waveform.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes what the b200 path computes; it does not apply to --impl reference")
    return a


def workload_config(a, n_gpus):
    secs = a.frames * 600 / SR
    return {
        "workload": "%s Decoder.forward(asr,F0_curve,N,s): %d utterances x %.1f s (T=%d frames) per GPU, "
                    "synthetic inputs, random-init weights (BASELINE.json configs[1])" % (a.variant, a.batch, secs, a.frames),
        "variant": a.variant, "batch_per_gpu": a.batch, "global_batch": a.batch * n_gpus, "frames": a.frames,
        "audio_seconds_per_step": a.batch * n_gpus * secs,
        "precision": {"fp32": "fp32 SIMT", "fp16": "tcgen05 fp16 operands, fp32 accumulate",
                      "bf16": "tcgen05 bf16 operands (generator.noise_res + front half on fp16 operands), fp32 accumulate"}[a.precision],
        "noise": "SineGen noise drawn on the device (Philox) inside the step",
        "l2": "L2 flushed between timed steps (256 MiB write); per-step working set >> 126 MB L2",
        "parallelism": ("replicas: utterances sharded per rank, no cross-rank math; every step's waveforms land in one preallocated "
                        "buffer on rank 0 -- --gather direct: the decoder's last kernel stores there over NVLink (symmetric memory), "
                        "--gather p2p (and the fallback): NCCL send / recv on a side stream that overlaps the next forward; all "
                        "transfers complete inside the timed region") if n_gpus > 1 else "single GPU",
    }


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference decoder restated on torch CPU kernels (oracle/decoder_torch.py), all host threads
# ------------------------------------------------------------------------------------------------
def cpu_reference_run(variant, frames, steps, warmup, batch=8):
    """The reference decoder on the host cores, `batch` utterances per step.  kind "reference": the unmodified Modules/
    staged under baseline/_ref by oracle/stage_reference.py; kind "port": oracle/decoder_torch.py (same ATen kernels)."""
    import torch
    from styletts2_lite_b200 import synth
    from styletts2_lite_b200.config import DecoderConfig
    # the CPU baseline leg is one of the places allowed to run the oracle / the staged reference
    from oracle import decoder_torch as O
    from oracle import stage_reference as SREF
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = DecoderConfig.hifigan() if variant == "hifigan" else DecoderConfig.istftnet()
    sd = synth.make_state_dict(cfg, 0, True)
    inp = synth.make_inputs(batch, frames, 1000, cfg, with_noise=False)
    ref = None
    try:
        ref = SREF.build_reference(cfg, sd)
    except Exception:  # noqa: BLE001
        ref = None
    if ref is not None:
        kind, what = "reference", "UNMODIFIED reference Modules/%s.py Decoder (staged under baseline/_ref), its own RNG draws" % cfg.type

        def fwd():
            with torch.no_grad():
                return ref(inp["asr"], inp["F0_curve"], inp["N"], inp["s"])
    else:
        kind, what = "port", ("torch-CPU port of the reference decoder (oracle/decoder_torch.py: the same ATen/oneDNN kernels the "
                              "reference dispatches to); baseline/_ref is not staged on this box")
        W = O.TorchWeights(sd)
        noise = torch.randn(batch, 600 * frames, 9)

        def fwd():
            return O.decoder_forward(W, cfg, inp["asr"], inp["F0_curve"], inp["N"], inp["s"], noise)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        out = fwd()
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    assert tuple(out.shape) == (batch, 1, 600 * frames) and bool(torch.isfinite(out).all())
    secs = batch * frames * 600 / SR
    mean = sum(times) / len(times)
    return {"value": secs / mean, "unit": UNIT, "cores": os.cpu_count(), "kind": kind,
            "sample": "%d utterances x %.1f s (T=%d) of the workload per step; %s; %d threads, %d steps after %d warm-up, "
                      "mean %.2f s/step" % (batch, frames * 600 / SR, frames, what, torch.get_num_threads(), steps, warmup, mean),
            "ms_per_step": mean * 1e3}


def run_reference(a, rank, world):
    if rank != 0:
        return None
    frames = a.cpu_frames or a.frames
    steps, warmup = a.steps, max(1, min(a.warmup, 1))
    r = cpu_reference_run(a.variant, frames, steps, warmup, batch=a.cpu_batch)
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": a.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(a, a.gpus),
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    return line


# ------------------------------------------------------------------------------------------------
# clocks sampler
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = str(gpu_index)
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) >= 8 and f[0] == self.idx:
                self.rows.append(f)

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:  # noqa: BLE001
                self.proc.kill()

    def summary(self):
        sm = sorted(float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()]
        reasons = []
        for name, col in (("hw_slowdown", 4), ("hw_thermal_slowdown", 5), ("sw_thermal_slowdown", 6), ("sw_power_cap", 7)):
            if any(r[col].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        pw = [float(r[3]) for r in self.rows if r[3].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows), "power_w_max": max(pw) if pw else None}


# DRAM bytes per launch of a kernel category, from the committed ncu launch list (profiles/<tag>_traffic.json,
# written by tools/summarize_profiles.py from `ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum`)
CATEGORY_KERNELS = {"conv_row": ("conv_row_kernel",), "conv_pipe": ("conv_pipe_kernel",), "conv_fused": ("conv_fused_kernel",), "conv_tc": ("conv_tc_kernel",),
                    "conv_simt": ("conv_simt_kernel",)}


def ncu_traffic(category):
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_traffic.json")))
    if not files or category not in CATEGORY_KERNELS:
        return None, None
    try:
        d = json.load(open(files[-1]))
        n = b = 0.0
        for name, k in d["kernels"].items():
            if any(t in name for t in CATEGORY_KERNELS[category]):
                n += k["launches"]
                b += k["launches"] * k["dram_bytes_per_launch"]
        return (b / n if n else None), os.path.relpath(files[-1], ROOT) + ": " + d.get("source", "")
    except (OSError, ValueError, KeyError):
        return None, None


# ------------------------------------------------------------------------------------------------
# auxiliary measurements (outside the timed region of the headline; none of them may break the main line)
# ------------------------------------------------------------------------------------------------
def _event_ms(torch, fn, warmup, iters):
    for i in range(warmup):
        fn(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        fn(warmup + i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def aux_cfg5(torch, dev, precision):
    """BASELINE configs[4]: iSTFTNet decoder, long-form 60 s utterances (8 per batch), one GPU, inputs resident."""
    from styletts2_lite_b200 import synth
    from styletts2_lite_b200.config import DecoderConfig
    from styletts2_lite_b200.decoder import B200Decoder
    cfg = DecoderConfig.istftnet()
    B, T = 8, 2400
    m = B200Decoder(cfg, precision)
    m.load_state_dict(synth.make_state_dict(cfg, 0, True))
    m = m.to(dev).eval()
    inp = {k: v.to(dev) for k, v in synth.make_inputs(B, T, seed=1005, cfg=cfg, with_noise=False).items()}
    out = [None]

    def fwd(i):
        with torch.no_grad():
            out[0] = m(inp["asr"], inp["F0_curve"], inp["N"], inp["s"], seed=77 + i)
    ms = _event_ms(torch, fwd, 2, 5)
    ok = tuple(out[0].shape) == (B, 1, 600 * T) and bool(torch.isfinite(out[0]).all())
    res = {"workload": "istftnet Decoder.forward, %d utterances x 60 s (T=%d), inputs resident" % (B, T), "precision": precision,
           "ms": round(ms, 3), "audio_s_per_s": round(B * 60.0 / (ms / 1e3), 1), "launches": int(m.last_launch_count()), "finite": ok}
    del m
    torch.cuda.empty_cache()
    return res


def aux_vocos(torch, dev, precision, B, T):
    """SURVEY 8(f) N4: the Vocos decoder variant (Modules/vocos.py) at the headline shape, inputs resident; next to it the
    unmodified reference module through PyTorch eager on the same GPU (fp32) when it is staged under baseline/_ref."""
    from styletts2_lite_b200 import synth
    from styletts2_lite_b200.config import DecoderConfig
    from styletts2_lite_b200.decoder import B200Decoder
    from oracle import stage_reference as SREF
    cfg = DecoderConfig.vocos()
    sd = synth.make_state_dict(cfg, 0, True)
    m = B200Decoder(cfg, precision)
    m.load_state_dict(sd)
    m = m.to(dev).eval()
    inp = {k: v.to(dev) for k, v in synth.make_inputs(B, T, seed=1006, cfg=cfg, with_noise=False).items()}
    out = [None]

    def fwd(i):
        with torch.no_grad():
            out[0] = m(inp["asr"], inp["F0_curve"], inp["N"], inp["s"])
    ms = _event_ms(torch, fwd, 3, 10)
    secs = B * T * 600 / 24000.0
    res = {"workload": "vocos Decoder.forward, %d utterances x %.0f s (T=%d), inputs resident" % (B, T * 600 / 24000.0, T),
           "precision": precision, "ms": round(ms, 3), "audio_s_per_s": round(secs / (ms / 1e3), 1),
           "launches": int(m.last_launch_count()),
           "finite": tuple(out[0].shape) == (B, 1, 600 * T) and bool(torch.isfinite(out[0]).all())}
    mine = out[0].float()
    del m
    torch.cuda.empty_cache()
    try:
        ref = SREF.build_reference(cfg, sd)
    except Exception:  # noqa: BLE001
        ref = None
    if ref is not None:
        ref = ref.to(dev)
        ro = [None]

        def rfwd(i):
            with torch.no_grad():
                ro[0] = ref(inp["asr"], inp["F0_curve"], inp["N"], inp["s"])
        rms = _event_ms(torch, rfwd, 2, 5)
        err = (ro[0].float() - mine)
        snr = 10.0 * float(torch.log10(ro[0].float().pow(2).sum() / err.pow(2).sum().clamp_min(1e-30)))
        res["eager_gpu_reference"] = {"kind": "reference", "precision": "fp32", "ms": round(rms, 3),
                                      "audio_s_per_s": round(secs / (rms / 1e3), 1), "snr_db_of_this_library_vs_it": round(snr, 1)}
        del ref
        torch.cuda.empty_cache()
    return res


def aux_eager_gpu(torch, dev, variant, B, T):
    """The pre-existing GPU path: the reference decoder through PyTorch eager (cuDNN / ATen kernels) on the same GPU and shape,
    fp32 and bf16 autocast.  The unmodified reference modules when staged (baseline/_ref), else the torch port of them."""
    from styletts2_lite_b200 import synth
    from styletts2_lite_b200.config import DecoderConfig
    from oracle import decoder_torch as O
    from oracle import stage_reference as SREF
    cfg = DecoderConfig.hifigan() if variant == "hifigan" else DecoderConfig.istftnet()
    sd = synth.make_state_dict(cfg, 0, True)
    inp = {k: v.to(dev) for k, v in synth.make_inputs(B, T, seed=1002, cfg=cfg, with_noise=False).items()}
    ref = None
    try:
        ref = SREF.build_reference(cfg, sd)
    except Exception:  # noqa: BLE001
        ref = None
    if ref is not None:
        ref = ref.to(dev)
        kind = "reference"

        def fwd(i):
            with torch.no_grad():
                return ref(inp["asr"], inp["F0_curve"], inp["N"], inp["s"])
    else:
        kind = "port"
        W = O.TorchWeights({k: v.to(dev) for k, v in sd.items()})
        noise = torch.randn(B, 600 * T, 9, device=dev)

        def fwd(i):
            return O.decoder_forward(W, cfg, inp["asr"], inp["F0_curve"], inp["N"], inp["s"], noise)
    res = {"kind": kind, "workload": "%s Decoder.forward through PyTorch eager on the GPU, %d x %.1f s" % (variant, B, T * 600 / SR)}
    secs = B * T * 600 / SR
    ms32 = _event_ms(torch, fwd, 1, 3)
    res["fp32"] = {"ms": round(ms32, 2), "audio_s_per_s": round(secs / (ms32 / 1e3), 1)}

    def fwd_bf16(i):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            return fwd(i)
    try:
        ms16 = _event_ms(torch, fwd_bf16, 1, 3)
        res["bf16_autocast"] = {"ms": round(ms16, 2), "audio_s_per_s": round(secs / (ms16 / 1e3), 1)}
    except Exception as ex:  # noqa: BLE001
        res["bf16_autocast"] = {"error": str(ex)[:200]}
    del ref
    torch.cuda.empty_cache()
    return res


def aux_cfg4(torch, dist, m, dev, rank, world, precision, direct=True):
    """BASELINE configs[3]: 1024 utterances x 10 s sharded over the ranks (parallel.shard_range), decoded in micro-batches of 32
    per rank, every micro-batch sent into its slice of ONE preallocated [1024,1,240000] buffer on rank 0 while the next one
    is being decoded (parallel.ShardedGather).  Timed on the device, max over ranks, second of two passes."""
    from styletts2_lite_b200 import synth
    from styletts2_lite_b200.parallel import ShardedGather
    N_UTT, T, MB = 1024, 400, 32
    S = 600 * T
    g = ShardedGather(N_UTT, S, MB, dev, direct=direct)
    inp = {k: v.to(dev) for k, v in synth.make_inputs(MB, T, seed=1004 + rank, cfg=m.cfg, with_noise=False).items()}
    mine = g.my_micro_batches()

    def one_pass(seed0):
        for j, (lo, hi) in enumerate(mine):
            n = hi - lo
            with torch.no_grad():
                out = m(inp["asr"][:n], inp["F0_curve"][:n], inp["N"][:n], inp["s"][:n], seed=seed0 + j, precision=precision,
                        out=g.target(j))
            g.submit(j, out)
        return g.finish()
    one_pass(100)                                    # warm-up pass (allocators, NCCL connections)
    dist.barrier()
    torch.cuda.synchronize()
    e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    e0.record()
    for j, (lo, hi) in enumerate(mine):
        n = hi - lo
        with torch.no_grad():
            out = m(inp["asr"][:n], inp["F0_curve"][:n], inp["N"][:n], inp["s"][:n], seed=5000 + j, precision=precision,
                    out=g.target(j))
        g.submit(j, out)
    e1.record()                                      # the last forward is issued; what follows is the exposed tail of the gather
    full = g.finish()
    e2.record()
    dist.barrier()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e2), e1.elapsed_time(e2)], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, tail_ms = float(t[0].item()), float(t[1].item())
    ok = True
    if rank == 0:
        ok = tuple(full.shape) == (N_UTT, 1, S) and bool(torch.isfinite(full[::97]).all())
    return {"workload": "hifigan Decoder, 1024 utterances x 10 s sharded over %d GPUs, micro-batches of %d, gathered to rank 0" % (world, MB),
            "utterances_per_rank": [hi - lo for lo, hi in g.spans], "micro_batches_per_rank": len(mine), "precision": precision,
            "ms": round(ms, 2), "audio_s_per_s": round(N_UTT * 10.0 / (ms / 1e3), 1),
            "gather_bytes_to_rank0": int((N_UTT - (g.spans[0][1] - g.spans[0][0])) * S * 4),
            "exposed_gather_tail_ms": round(tail_ms, 3), "finite": ok,
            "gather": ("direct: the decoder's last kernel stores into rank 0's buffer (symmetric memory over NVLink)" if g.direct
                       else "p2p: NCCL send / recv on a side stream"),
            "limiter": "rank 0 ingests (world-1)/world of 983 MB over its NVLink ports while it decodes its own shard; only the "
                       "tail after the last forward (exposed_gather_tail_ms) is not hidden"}


DUMP_BYTES = 64 << 20


def dump_waveform(out_dir, wave):
    """DIR/waveform.npy: float32 [B,1,S]; above DUMP_BYTES, a seeded sample of utterances (and of leading samples if a single
    utterance is larger), the same one for the same arguments."""
    import numpy as np
    import torch
    n, row_bytes = wave.shape[0], wave[0].numel() * 4
    keep = max(1, min(n, DUMP_BYTES // row_bytes))
    if keep < n:
        rows = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        wave = wave[torch.from_numpy(rows).to(wave.device)]
    wave = wave[..., :DUMP_BYTES // 4]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "waveform.npy"), wave.float().cpu().numpy())


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def run_b200(a, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    from styletts2_lite_b200 import synth
    from styletts2_lite_b200.config import DecoderConfig
    from styletts2_lite_b200.decoder import B200Decoder
    from styletts2_lite_b200.parallel import ShardedGather

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg = DecoderConfig.hifigan() if a.variant == "hifigan" else DecoderConfig.istftnet()
    B, T = a.batch, a.frames
    S = 600 * T
    m = B200Decoder(cfg, a.precision)
    m.load_state_dict(synth.make_state_dict(cfg, 0, True))
    m = m.to(dev).eval()
    inp = synth.make_inputs(B, T, seed=1000 + 2 + rank, cfg=cfg, with_noise=False)
    host = {k: v.pin_memory() for k, v in inp.items()}
    res = {k: v.to(dev) for k, v in inp.items()}
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # N > 1: one job = world x B utterances, one micro-batch per rank per step, straight into rank 0's preallocated buffer
    gatherer = ShardedGather(B * world, S, B, dev, direct=(a.gather == "direct")) if world > 1 else None
    gather_calls = [0]

    def submit_gather(out):
        gatherer.submit(0, out)
        gather_calls[0] += 1
        if gather_calls[0] % 8 == 0:                 # bound the number of in-flight sends (their sources are kept alive)
            gatherer.finish()

    def step_resident(i):
        with torch.no_grad():
            out = m(res["asr"], res["F0_curve"], res["N"], res["s"], seed=1234 + i,
                    out=(gatherer.target(0) if gatherer is not None else None))
        if world > 1:
            submit_gather(out)
        return out

    # end to end through the package's host-fed serving loop (styletts2_lite_b200/streaming.py): every step copies its
    # inputs from pinned host memory and its waveform back to pinned host memory; the copies of neighbouring steps
    # overlap the decoder on separate streams
    from styletts2_lite_b200.streaming import PipelinedDecoder
    pipe = PipelinedDecoder(m, dev, after_forward=(submit_gather if world > 1 else None))

    def run_e2e(steps, first_seed):
        seeds = iter(range(first_seed, first_seed + steps))
        last = None
        for wav in pipe.decode((host for _ in range(steps)), seeds):
            last = wav
        if gatherer is not None:
            gatherer.finish()
        return last

    def timed(fn, steps, warmup):
        for i in range(warmup):
            fn(i)
        if gatherer is not None:
            gatherer.finish()
        barrier()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        t_wall = time.perf_counter()
        out = None
        for i in range(steps):
            flush.fill_(i & 0xFF)                    # L2 flush, outside the event pair
            evs[i][0].record()
            out = fn(warmup + i)
            if gatherer is not None and i == steps - 1:
                gatherer.finish()                    # every gather of the timed steps completes inside the last event pair
            evs[i][1].record()
        barrier()
        wall = time.perf_counter() - t_wall
        ms = [s.elapsed_time(e) for s, e in evs]
        total = torch.tensor([sum(ms)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(total, op=dist.ReduceOp.MAX)
        return float(total.item()), ms, wall, out

    sampler = ClockSampler(local_rank)
    sampler.start()
    total_ms, per_step, wall, last = timed(step_resident, a.steps, a.warmup)
    clocks = sampler.summary()
    sampler.stop()
    launches = m.last_launch_count()
    if a.dump_outputs:
        # what a caller of the timed path holds after its last step: N > 1 gathers every rank's waveforms on rank 0
        wave = gatherer.finish() if gatherer is not None else last
        if rank == 0:
            dump_waveform(a.dump_outputs, wave)
        barrier()                                    # no rank writes into rank 0's buffer again before it is read
    last = None
    run_e2e(max(2, a.warmup // 2 + 1), 4000)                  # warm-up
    barrier()
    t_e2e = time.perf_counter()                                # host clock: the loop ends with every waveform on the host
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    wav = run_e2e(a.steps, 4321)
    e1.record()
    barrier()
    wall_e2e_ms = (time.perf_counter() - t_e2e) * 1e3
    assert wav is not None and tuple(wav.shape) == (B, 1, S) and bool(torch.isfinite(wav).all())
    te = torch.tensor([max(e0.elapsed_time(e1), 0.0), wall_e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    total_e2e_ms = float(te[1].item())                         # wall clock >= device time; it includes the last D2H

    # per-category event profile (same workload, profiling on) -> roofline of the dominant kernel
    m.set_profiling(True)
    prof_acc = None
    for i in range(a.steps):
        step_resident(10_000 + i)
        p = m.get_profile()
        if prof_acc is None:
            prof_acc = p
        else:
            for c in p:
                for k in p[c]:
                    prof_acc[c][k] += p[c][k]
    m.set_profiling(False)
    if gatherer is not None:
        gatherer.finish()
    torch.cuda.synchronize()

    audio_s = B * world * S / SR
    ms_per_step = total_ms / a.steps
    value = audio_s / (ms_per_step / 1e3)
    e2e_value = audio_s / (total_e2e_ms / a.steps / 1e3)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except (OSError, ValueError):
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    tc_peak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1590.0)))
    peak_src = "MEASURED_PEAKS.json (sustained bf16, copy HBM)" if peaks else "fallback (B200_PROFILING.md)"
    kernels = {}
    prof_ms_step = 0.0
    for c, v in prof_acc.items():
        if v["launches"] == 0:
            continue
        ms_c = v["ms"] / a.steps
        prof_ms_step += ms_c
        kernels[c] = {"ms_per_step": round(ms_c, 4), "launches_per_step": v["launches"] // a.steps,
                      "tflops": round(v["flops"] / v["ms"] / 1e9, 2) if v["flops"] and v["ms"] else None,
                      "gbs": round(v["bytes"] / v["ms"] / 1e6, 1) if v["bytes"] and v["ms"] else None}
    for c in kernels:
        kernels[c]["share"] = round(kernels[c]["ms_per_step"] / prof_ms_step, 4)
    dom = max(kernels, key=lambda c: kernels[c]["ms_per_step"])
    if dom in ("conv_tc", "conv_simt", "conv_fused"):
        v = prof_acc[dom]
        achieved = v["flops"] / v["ms"] / 1e9
        roof = {"kernel": dom, "bound": "tensor", "achieved": achieved, "peak": tc_peak, "unit": "TFLOP/s",
                "frac": achieved / tc_peak, "traffic": None}
    else:
        v = prof_acc[dom]
        achieved = v["bytes"] / v["ms"] / 1e6
        roof = {"kernel": dom, "bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                "frac": achieved / hbm_peak, "traffic": None}
    roof["traffic"], roof["traffic_source"] = ncu_traffic(dom)
    roof["algorithmic_bytes_per_launch"] = prof_acc[dom]["bytes"] / max(prof_acc[dom]["launches"], 1)
    roof["avg_launch_ms"] = prof_acc[dom]["ms"] / max(prof_acc[dom]["launches"], 1)
    roof["peak_source"] = peak_src
    roof["kernels"] = kernels
    roof["profiled_ms_per_step"] = round(prof_ms_step, 3)
    # the HBM-bound half, always reported next to the dominant kernel
    if "affine_act" in prof_acc and prof_acc["affine_act"]["ms"] > 0:
        g = prof_acc["affine_act"]["bytes"] / prof_acc["affine_act"]["ms"] / 1e6
        roof["affine_act_hbm"] = {"achieved": g, "peak": hbm_peak, "unit": "GB/s", "frac": g / hbm_peak}

    cfg4 = None
    if world > 1 and not a.no_aux and a.precision != "fp32" and a.variant == "hifigan":
        # BASELINE configs[3] on every rank (a collective job); after the headline's timed regions
        try:
            cfg4 = aux_cfg4(torch, dist, m, dev, rank, world, a.precision, direct=(a.gather == "direct"))
        except Exception as ex:  # noqa: BLE001
            cfg4 = {"error": str(ex)[:300]}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return None
    h2d = sum(host[k].numel() * 4 for k in ("asr", "F0_curve", "N", "s"))
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"fp32": "f32", "bf16": "bf16", "fp16": "f16"}[a.precision], "data": "synthetic",
            "config": workload_config(a, world),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": B * S * 4,
                    "ms_per_step": total_e2e_ms / a.steps,
                    "how": "styletts2_lite_b200.streaming.PipelinedDecoder over %d host batches (pinned H2D, forward, pinned D2H "
                           "every step; copies overlap the neighbouring forwards); host wall clock, max over ranks" % a.steps},
            "gpu_launches": int(launches * a.steps), "launches_per_step": int(launches),
            "clocks": clocks, "roofline": roof, "wall_s_timed_region": round(wall, 3),
            "per_step_ms": [round(x, 3) for x in per_step]}
    if gatherer is not None:
        line["config"]["gather_used"] = "direct (symmetric memory)" if gatherer.direct else "p2p (NCCL send / recv)"
    if world == 1 and not a.no_cpu_baseline:
        r = cpu_reference_run(a.variant, a.cpu_frames or a.frames, 2, 1, batch=a.cpu_batch)
        line["cpu_baseline"] = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
    if cfg4 is not None:
        line["cfg4_sharded_1024x10s"] = cfg4
    aux_on = not a.no_aux and a.precision != "fp32"
    if world == 1 and aux_on and not a.no_cpu_baseline and not a.no_chain:
        # auxiliary, outside the timed region: BASELINE configs[2] (32 x 8 s, token ids -> waveform through the TextEncoder,
        # the prosody predictor, the length regulator and the Decoder of this library); never allowed to break the main line
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            from bench_chain import run_chain
            line["full_path_cfg3"] = run_chain(32, 64, 320, a.precision, 5)
        except Exception as ex:  # noqa: BLE001
            line["full_path_cfg3"] = {"error": str(ex)[:300]}
    if world == 1 and aux_on:
        del m
        torch.cuda.empty_cache()
        for key, fn in (("cfg5_istftnet_60s", lambda: aux_cfg5(torch, dev, a.precision)),
                        ("vocos_n4", lambda: aux_vocos(torch, dev, a.precision, B, T)),
                        ("eager_gpu", lambda: aux_eager_gpu(torch, dev, a.variant, B, T))):
            try:
                line[key] = fn()
            except Exception as ex:  # noqa: BLE001
                line[key] = {"error": str(ex)[:300]}
                torch.cuda.empty_cache()
    if world > 1:
        dist.destroy_process_group()
    return line


class _StdoutToStderr:
    """Library banners (e.g. "NCCL version ..." on stdout) must not mix with the one JSON line: while active, file descriptor 1
    points at stderr; the JSON line is printed after restore()."""

    def __init__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)

    def restore(self):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


def main():
    a = parse()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    guard = _StdoutToStderr()
    line = run_reference(a, rank, world) if a.impl == "reference" else run_b200(a, rank, local_rank, world)
    guard.restore()
    if line is not None:
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
