"""Drop-in `Decoder` modules for the StyleTTS2-lite waveform decoder.

Host-side mirror of the reference interface (Modules/hifigan.py:416-475 and
Modules/istftnet.py:660-721): same constructor keywords, same `state_dict` keys
(legacy weight-norm pairs, so `load_state_dict` of a reference checkpoint works,
inference.py:160), same `forward(asr, F0_curve, N, s) -> [B,1,600*T]`.  The
arithmetic runs in the sm_100a kernels behind include/st2_b200.h; PyTorch only
owns the tensors, the stream and the workspace.  There is no CPU path.
"""
from __future__ import annotations

import collections

import ctypes as C
from typing import Dict, Optional

import torch
import torch.nn as nn

from . import _lib
from .config import DecoderConfig, buffer_specs, param_specs
from .synth import stft_buffers


def _register(root: nn.Module, name: str, tensor: torch.Tensor, buffer: bool = False) -> None:
    parts = name.split(".")
    mod = root
    for p in parts[:-1]:
        if p not in mod._modules:
            mod.add_module(p, nn.Module())
        mod = mod._modules[p]
    if buffer:
        mod.register_buffer(parts[-1], tensor)
    else:
        mod.register_parameter(parts[-1], nn.Parameter(tensor, requires_grad=False))


class B200Decoder(nn.Module):
    """Base of the drop-in decoders (hifigan, istftnet, vocos).  `precision`: 'fp32' (SIMT, <=1e-4 of the CPU
    reference), 'bf16' (tcgen05, bf16 operands; generator.noise_res on fp16 operands) or
    'fp16' (tcgen05, fp16 operands)."""

    def __init__(self, cfg: DecoderConfig, precision: str = "fp32", fp16_storage: bool = True):
        super().__init__()
        self.fp16_storage = fp16_storage        # 16-bit precisions: stage-private generator tensors in fp16 (DESIGN.md section 3)
        if precision not in _lib.PREC:
            raise ValueError("precision must be one of %s" % list(_lib.PREC))
        self.cfg = cfg
        self.precision = precision
        for name, shape, kind in param_specs(cfg):
            init = torch.ones(shape) if kind in ("alpha", "gamma") else torch.zeros(shape)
            _register(self, name, init)
        if cfg.is_vocos:
            _register(self, "generator.stft.istft.window", torch.hann_window(cfg.gen_istft_n_fft), buffer=True)   # vocos.py:192-193
        elif cfg.is_istft:
            bufs = stft_buffers(cfg)
            for name, _ in buffer_specs(cfg):
                _register(self, name, bufs[name].clone(), buffer=True)
        self._handle: Optional[C.c_void_p] = None
        self._dirty = True
        self._workspace: Optional[torch.Tensor] = None
        self._taps: Dict[str, torch.Tensor] = {}
        self._graphs: "collections.OrderedDict[tuple, dict]" = collections.OrderedDict()   # LRU: newest last
        self.max_graphs = 8                     # each captured shape owns a private workspace + static I/O: bound the cache
        self._ws_bytes: Dict[tuple, int] = {}   # (B, T, precision, plan) -> workspace bytes (the host dry run costs ~0.1 ms)
        self._option_generation = 0             # bumped by set_option(): part of the plan key of both caches
        self._profiling = False
        self.train(False)

    # ---- weights -------------------------------------------------------------------------
    def _apply(self, fn, *a, **k):
        r = super()._apply(fn, *a, **k)
        self._dirty = True
        self._graphs.clear()
        return r

    def load_state_dict(self, state_dict, strict: bool = True, *a, **k):
        r = super().load_state_dict(state_dict, strict, *a, **k)
        self._dirty = True
        return r

    def refresh_weights(self) -> None:
        """Re-pack after an in-place parameter update."""
        self._dirty = True
        self._graphs.clear()

    def _sync(self, device: torch.device) -> None:
        lib = _lib.load()
        self._graphs.clear()                      # finalize re-allocates the packed weights captured graphs point to
        self._ws_bytes.clear()
        if self._handle is None:
            h = C.c_void_p()
            cc = _lib.St2Config.from_config(self.cfg)
            _lib.check(lib.st2_decoder_create(C.byref(cc), C.byref(h)), "st2_decoder_create")
            self._handle = h
        _lib.check(lib.st2_decoder_set_option(self._handle, b"fp16_storage", 1 if self.fp16_storage else 0), "set_option")
        keep = []
        for name, t in self.state_dict().items():
            if t.device != device:
                raise _lib.St2Error("parameter %s is on %s but inputs are on %s; call .to(device)" % (name, t.device, device))
            t = t.detach().float().contiguous()
            keep.append(t)
            shape = (C.c_int64 * max(t.dim(), 1))(*t.shape)
            _lib.check(lib.st2_decoder_set_weight(self._handle, name.encode(), _lib.ptr(t), shape, t.dim()),
                       "st2_decoder_set_weight(%s)" % name)
        stream = torch.cuda.current_stream(device).cuda_stream
        _lib.check(lib.st2_decoder_finalize(self._handle, C.c_void_p(stream)), "st2_decoder_finalize")
        del keep
        self._dirty = False

    def num_params(self) -> int:
        return sum(p.numel() for p in self.parameters())

    def set_option(self, name: str, value: int) -> None:
        """st2_decoder_set_option on this module's handle ("fp16_xt", "fp16_run", ...: INTEGRATION.md section 3e).  The next
        forward plans its workspace and captures its CUDA graph again."""
        if self._handle is None:
            self._sync(next(self.parameters()).device)
        _lib.check(_lib.load().st2_decoder_set_option(self._handle, name.encode(), int(value)), "set_option(%s)" % name)
        self._option_generation += 1

    def _plan_key(self) -> tuple:
        # the switches that decide the kernel plan, and with it the workspace size and the launches a graph captures
        return (_lib.tuning_generation(), self._option_generation)

    # ---- forward ---------------------------------------------------------------------------
    def workspace_bytes(self, B: int, T: int, precision: Optional[str] = None) -> int:
        lib = _lib.load()
        n = lib.st2_decoder_workspace_bytes(self._handle, B, T, _lib.PREC[precision or self.precision])
        return _lib.check(n, "st2_decoder_workspace_bytes")

    def set_tap(self, name: str, B: int, rows: int, C_: int) -> torch.Tensor:
        """Register a debug tap; returns the [B, rows, C] buffer the next forward fills."""
        dev = next(self.parameters()).device
        buf = torch.zeros(B, rows, C_, device=dev, dtype=torch.float32)
        if self._handle is None:
            self._sync(dev)
        _lib.check(_lib.load().st2_decoder_set_tap(self._handle, name.encode(), _lib.ptr(buf), buf.numel()), "set_tap")
        self._taps[name] = buf
        return buf

    def clear_taps(self) -> None:
        for name in list(self._taps):
            _lib.load().st2_decoder_set_tap(self._handle, name.encode(), None, 0)
        self._taps.clear()

    # ---- CUDA-graph replay for small batches ------------------------------------------------
    def _forward_graph(self, asr, F0_curve, N, s, seed, prec_name):
        """One captured graph per (B, T, precision, device, switches): the ~270 launches of a forward replay as one graph
        launch.  Inputs are copied into the graph's static buffers, the Philox seed lives in device memory
        (st2_decoder_set_seed_buffer), the returned waveform is a copy of the static output."""
        lib = _lib.load()
        dev = asr.device
        B, _, T = asr.shape
        prec = _lib.PREC[prec_name]
        key = (B, T, prec, dev.index) + self._plan_key()
        g = self._graphs.get(key)
        if g is not None:
            self._graphs.move_to_end(key)
        if g is None:
            while len(self._graphs) >= max(1, self.max_graphs):       # least recently used shape goes (frees its workspace)
                self._graphs.popitem(last=False)
            S = self.cfg.samples_per_frame * T
            need = self._workspace_need(B, T, prec)
            g = {"asr": torch.empty(B, self.cfg.dim_in, T, device=dev), "f0": torch.empty(B, 2 * T, device=dev),
                 "n": torch.empty(B, 2 * T, device=dev), "s": torch.empty(B, self.cfg.style_dim, device=dev),
                 "seed": torch.zeros(1, dtype=torch.int64, device=dev), "out": torch.empty(B, 1, S, device=dev),
                 "ws": torch.empty(need, dtype=torch.uint8, device=dev)}
            for k_, t in (("asr", asr), ("f0", F0_curve), ("n", N), ("s", s)):
                g[k_].copy_(t)

            def launch():
                stream = torch.cuda.current_stream(dev).cuda_stream
                _lib.check(lib.st2_decoder_forward(self._handle, _lib.ptr(g["asr"]), _lib.ptr(g["f0"]), _lib.ptr(g["n"]),
                                                   _lib.ptr(g["s"]), None, C.c_uint64(0), _lib.ptr(g["out"]), B, T, prec,
                                                   _lib.ptr(g["ws"]), g["ws"].numel(), C.c_void_p(stream)),
                           "st2_decoder_forward (graph capture)")

            _lib.check(lib.st2_decoder_set_seed_buffer(self._handle, _lib.ptr(g["seed"])), "set_seed_buffer")
            try:
                side = torch.cuda.Stream(device=dev)
                side.wait_stream(torch.cuda.current_stream(dev))
                with torch.cuda.stream(side):
                    launch()                                    # eager warm-up (function attributes, tensor-map driver entry)
                torch.cuda.current_stream(dev).wait_stream(side)
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    launch()
            finally:
                lib.st2_decoder_set_seed_buffer(self._handle, None)
            g["graph"] = graph
            self._graphs[key] = g
        for k_, t in (("asr", asr), ("f0", F0_curve), ("n", N), ("s", s)):
            g[k_].copy_(t, non_blocking=True)
        g["seed"].fill_(seed - (1 << 64) if seed >= (1 << 63) else seed)
        g["graph"].replay()
        return g["out"].clone()

    def forward(self, asr, F0_curve, N, s, noise: Optional[torch.Tensor] = None, seed: Optional[int] = None,
                precision: Optional[str] = None, cuda_graph: bool = False, out: Optional[torch.Tensor] = None):
        """`out` (optional): a contiguous fp32 [B,1,S] CUDA tensor the waveform is written into -- it may live on another GPU
        of the box (peer memory, e.g. `parallel.ShardedGather.target()`): the last kernel of the forward then stores over NVLink
        straight into the gathered buffer."""
        if self.training:
            raise RuntimeError("B200Decoder is inference-only (the reference's training-time F0/N smoothing, "
                               "hifigan.py:447-455, is out of scope); call .eval()")
        if not asr.is_cuda:
            raise _lib.St2Error("B200Decoder has no CPU path: inputs must be CUDA tensors")
        lib = _lib.load()
        dev = asr.device
        B, Cin, T = asr.shape
        if Cin != self.cfg.dim_in or F0_curve.shape != (B, 2 * T) or N.shape != (B, 2 * T) or s.shape != (B, self.cfg.style_dim):
            raise ValueError("expected asr [B,%d,T], F0_curve [B,2T], N [B,2T], s [B,%d]; got %s %s %s %s" %
                             (self.cfg.dim_in, self.cfg.style_dim, tuple(asr.shape), tuple(F0_curve.shape),
                              tuple(N.shape), tuple(s.shape)))
        prec = _lib.PREC[precision or self.precision]
        with torch.cuda.device(dev):
            if self._dirty or self._handle is None:
                self._sync(dev)
            asr_, f0_, n_, s_ = (t.detach().float().contiguous() for t in (asr, F0_curve, N, s))
            S = self.cfg.samples_per_frame * T
            noise_ = None
            if noise is not None:
                if tuple(noise.shape) != (B, S, 9):
                    raise ValueError("noise must be [B,%d,9]" % S)
                noise_ = noise.detach().float().contiguous()
            if seed is None:
                seed = int(torch.randint(0, 2 ** 62, (1,)).item())      # global torch RNG, like the reference
            # graph replay needs a launch sequence without host-side state: not with taps, a noise tape or the per-launch
            # event profile (its cudaEventRecord calls would be captured and later read back as garbage) -> eager
            if cuda_graph and noise_ is None and not self._taps and not self._profiling and out is None:
                return self._forward_graph(asr_, f0_, n_, s_, seed, precision or self.precision)
            need = self._workspace_need(B, T, prec)
            if self._workspace is None or self._workspace.numel() < need or self._workspace.device != dev:
                self._workspace = None
                self._workspace = torch.empty(need, dtype=torch.uint8, device=dev)
            if out is None:
                out = torch.empty(B, 1, S, dtype=torch.float32, device=dev)
            elif tuple(out.shape) != (B, 1, S) or out.dtype != torch.float32 or not out.is_cuda or not out.is_contiguous():
                raise ValueError("out must be a contiguous float32 CUDA tensor of shape [%d,1,%d]" % (B, S))
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(lib.st2_decoder_forward(self._handle, _lib.ptr(asr_), _lib.ptr(f0_), _lib.ptr(n_), _lib.ptr(s_),
                                               _lib.ptr(noise_), C.c_uint64(seed), _lib.ptr(out), B, T, prec,
                                               _lib.ptr(self._workspace), self._workspace.numel(),
                                               C.c_void_p(stream)), "st2_decoder_forward")
        return out

    def _workspace_need(self, B: int, T: int, prec: int) -> int:
        key = (B, T, prec) + self._plan_key()
        n = self._ws_bytes.get(key)
        if n is None:
            n = _lib.check(_lib.load().st2_decoder_workspace_bytes(self._handle, B, T, prec), "st2_decoder_workspace_bytes")
            if len(self._ws_bytes) > 256:
                self._ws_bytes.clear()
            self._ws_bytes[key] = n
        return n

    def set_profiling(self, enable: bool) -> None:
        """Per-launch CUDA-event profile of the following forwards (bench.py's roofline leg)."""
        if self._handle is None:
            self._sync(next(self.parameters()).device)
        _lib.check(_lib.load().st2_decoder_set_profiling(self._handle, 1 if enable else 0), "set_profiling")
        self._profiling = bool(enable)

    def get_profile(self) -> Dict[str, Dict[str, float]]:
        """{category: {ms, launches, flops, bytes}} of the last profiled forward (waits for it)."""
        lib = _lib.load()
        n = lib.st2_profile_num_categories()
        ms, fl, by = (C.c_double * n)(), (C.c_double * n)(), (C.c_double * n)()
        ln = (C.c_int64 * n)()
        _lib.check(lib.st2_decoder_get_profile(self._handle, ms, ln, fl, by), "get_profile")
        return {lib.st2_profile_category_name(i).decode(): {"ms": ms[i], "launches": int(ln[i]), "flops": fl[i],
                                                            "bytes": by[i]} for i in range(n)}

    def get_profile_launches(self, max_n: int = 4096):
        """[(category, ms, flops, bytes)] per launch of the last profiled forward, in launch order."""
        lib = _lib.load()
        cat, ms = (C.c_int32 * max_n)(), (C.c_float * max_n)()
        fl, by = (C.c_double * max_n)(), (C.c_double * max_n)()
        n = _lib.check(lib.st2_decoder_get_profile_launches(self._handle, max_n, cat, ms, fl, by), "get_profile_launches")
        return [(lib.st2_profile_category_name(cat[i]).decode(), ms[i], fl[i], by[i]) for i in range(n)]

    def last_launch_count(self) -> int:
        return int(_lib.load().st2_decoder_last_launch_count(self._handle)) if self._handle else 0

    def __del__(self):
        try:
            if self._handle is not None:
                _lib.load().st2_decoder_destroy(self._handle)
                self._handle = None
        except Exception:
            pass
