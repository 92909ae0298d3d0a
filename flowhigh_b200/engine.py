"""Host-side orchestration of the FLowHigh hot path on one B200.

Python here only owns buffers (torch tensors as device memory), packs weights once, and
sequences kernel launches through the C ABI (flowhigh_b200/_lib.py).  No torch operator runs
on the per-clip path: every stage of `FlowHighSR.generate` (flowhighsr.py:51-102) is one of
the hand-written kernels.

Two numeric modes:
  * precision='fp32' -- CUDA-core fp32 kernels on the reference's layouts; the parity path
    (waveform max-abs <= 1e-4 / mel L1 <= 1e-4 against the reference's fp32 implementation).
  * precision='bf16' | 'fp16' -- tcgen05/TMEM implicit-GEMM kernels on chunked 16-bit operands with
    fp32 accumulators and an fp32 residual stream; the throughput path.  Both formats run at the
    same tensor rate and move the same bytes; IEEE half carries 3 more mantissa bits, which is what
    the LSD <= 0.05 dB bar needs (every GEMM input here is O(1)-O(10^2): far inside fp16 range).
"""
from __future__ import annotations

import collections
import contextlib
from os import environ as _environ
_os_environ_get = _environ.get
import ctypes as C
import math
from typing import Dict, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib, packing, rk, tables
from .config import BackboneConfig, MelConfig, VocoderConfig
from .weights import FH, VOC

HALO = 32  # zero rows on each side of a chunked vocoder sequence (>= max dilated reach 25)


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


class _TcWeight:
    __slots__ = ("packed", "bias", "off", "off_c", "P", "ntaps", "cin", "cout", "cin_pad", "cout_pad", "bn", "two_cta")


class _F32Weight:
    __slots__ = ("w", "off", "bias", "P", "ntaps", "cin", "cout")


class Engine:
    def __init__(self, sd: Dict[str, torch.Tensor], vcfg: VocoderConfig, bcfg: BackboneConfig = BackboneConfig(),
                 device="cuda:0", precision: str = "fp16", precise_mel: Optional[bool] = None):
        if precision not in ("fp32", "bf16", "fp16", "fp16x2"):
            raise ValueError("precision must be 'fp32', 'bf16', 'fp16' or 'fp16x2'")
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("flowhigh_b200 has no CPU path: a CUDA (sm_100a) device is required")
        vcfg.validate()
        self.lib = _lib.load()
        self.vcfg, self.bcfg, self.mcfg = vcfg, bcfg, MelConfig()
        self.precision = precision
        self.tc = precision in ("bf16", "fp16", "fp16x2")
        self.fp16 = 1 if precision in ("fp16", "fp16x2") else 0
        # "fp16x2": the vocoder's activation operands are hi + lo fp16 pairs against duplicated weights (twice the MMAs,
        # ~22-bit activations).  tools/lsd_emulation.py: activation rounding, not weight rounding, sets the log-spectral
        # distance of the 16-bit path (0.093 of 0.094 dB on the high-dynamic-range fixture); this mode removes it.
        self.split = precision == "fp16x2"
        self.h16 = torch.float16 if self.fp16 else torch.bfloat16  # storage dtype of MMA operands
        self.k16 = 2 if self.fp16 else 1                          # out_mode / out_kind code of that dtype
        self.precise_mel = (precision == "fp32") if precise_mel is None else precise_mel
        # persistent scratch buffers, keyed by (name, exact shape, dtype), least recently used first.  The cache is
        # capped (FH_BUF_CAP_GB, default 120 of the 180 GB): a service that sees ever new clip lengths evicts the buffers
        # of old shapes instead of growing without bound.  CUDA graphs keep their own references (touch log below).
        self._bufs: "collections.OrderedDict[tuple, torch.Tensor]" = collections.OrderedDict()
        self._buf_bytes = 0
        self._buf_cap = int(float(_os_environ_get("FH_BUF_CAP_GB", "120")) * (1 << 30))
        self._buf_epoch = 0            # bumped per top-level call: buffers touched in the current call are never evicted
        self._buf_last: Dict[tuple, int] = {}
        self._touch_log = None         # {id: object} while a CUDA graph is warmed up / captured: what the graph must keep alive
        self.profile = None
        import os as _os
        self._cool_ms = float(_os.environ.get("FH_PROFILE_COOL_MS", "0"))
        # fp16 path: the first convolution of an AMP unit writes fp16 rows and the snake behind it reads them as MMA
        # operands (fh_snake_aa_chunked_h) -- the fp32 round trip of that tensor disappears
        self.y16 = self.fp16 and not self.split
        # AMP branches of a stage on parallel streams for small batches (B = 1 latency path)
        self.branch_streams = True
        self.branch_streams_max_batch = 4
        self._branch_streams = []
        self._time_cache: "collections.OrderedDict[float, dict]" = collections.OrderedDict()  # LRU, <= 512 grid values
        dev = self.device
        with torch.cuda.device(dev):
            self.sd = {k: v.detach().to(dev, torch.float32).contiguous() for k, v in sd.items()}
            # ---- DSP tables
            self.window = torch.hann_window(2048, dtype=torch.float32).to(dev)
            self.twiddle = torch.from_numpy(tables.fft_twiddles()).to(dev)
            ms, ml, mw, self.mel_stride = tables.mel_filterbank_sparse()
            self.mel_start = torch.from_numpy(ms).to(dev)
            self.mel_len = torch.from_numpy(ml).to(dev)
            self.mel_w = torch.from_numpy(mw).to(dev)
            self._resample_taps: Dict[tuple, tuple] = {}
            # overflow / NaN guard of the 16-bit path (include/flowhigh_b200.h fh_set_status_word): one device word,
            # reset at the start of a pipeline, copied to pinned host memory at its end, read once per generate()
            self.status = torch.zeros(1, dtype=torch.int32, device=dev)
            self._status_host = torch.zeros(1, dtype=torch.int32).pin_memory()
            self._prep_backbone()
            self._prep_vocoder()
        torch.cuda.synchronize(dev)
        self._bind_status()

    # ------------------------------------------------------------------ plumbing
    @property
    def stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def new_call(self):
        """Marks the start of a top-level call (generate_batch / bench step): buffers last used by earlier calls
        become evictable when the cache cap is hit, and the calling thread's launches report to this engine's
        status word."""
        self._buf_epoch += 1
        self._bind_status()

    _status_owner = None  # id of the engine whose status word the library currently holds (this thread)

    def _bind_status(self):
        _lib.check(self.lib.fh_set_status_word(self.status.data_ptr()), "fh_set_status_word")
        Engine._status_owner = id(self)

    def __del__(self):
        # never leave the library pointing at a status word that is about to be freed
        try:
            if Engine._status_owner == id(self):
                self.lib.fh_set_status_word(None)
                Engine._status_owner = None
        except Exception:  # interpreter shutdown
            pass

    def status_begin(self):
        """Zeroes the status word (stream-ordered; capturable)."""
        self._call("fh_fill_u32", self.status.data_ptr(), 0, 1, self.stream)

    def status_end(self):
        """Stream-ordered copy of the status word to pinned host memory (capturable)."""
        self._status_host.copy_(self.status, non_blocking=True)

    def status_read(self) -> int:
        """Synchronises the current stream and returns the status word of the last status_begin/status_end bracket:
        bit 0 = a 16-bit operand saturated (fp16 |x| >= 65504) or was inf / NaN."""
        torch.cuda.current_stream(self.device).synchronize()
        return int(self._status_host[0])

    def _evict_for(self, need: int):
        if torch.cuda.is_current_stream_capturing():
            return
        for key in list(self._bufs.keys()):
            if self._buf_bytes + need <= self._buf_cap:
                break
            if self._buf_last.get(key, -1) >= self._buf_epoch:
                continue  # in use by the current call
            t = self._bufs.pop(key)
            self._buf_last.pop(key, None)
            self._buf_bytes -= t.numel() * t.element_size()

    def buf(self, name: str, shape, dtype=torch.float32, zero: bool = True) -> torch.Tensor:
        key = (name, tuple(int(s) for s in shape), dtype)
        t = self._bufs.get(key)
        self._buf_last[key] = self._buf_epoch
        if t is not None:
            self._bufs.move_to_end(key)
        if t is None:
            need = int(np.prod(key[1], dtype=np.int64)) * torch.empty((), dtype=dtype).element_size()
            if self._buf_bytes + need > self._buf_cap:
                self._evict_for(need)
            t = (torch.zeros if zero else torch.empty)(key[1], dtype=dtype, device=self.device)
            self._bufs[key] = t
            self._buf_bytes += need
            # The zero-fill runs on the stream that is current NOW, but the buffer may first be used on another one
            # (the AMP branch streams wait on an event recorded before their scratch buffers are created): without
            # this, the fill can land after a branch kernel has written the buffer.  First use of a shape only.
            if not torch.cuda.is_current_stream_capturing():
                torch.cuda.current_stream(self.device).synchronize()
        if self._touch_log is not None:
            self._touch_log[id(t)] = t
        return t

    def _chk(self, *tensors):
        """Kernels take raw pointers: every tensor handed to the engine must be dense fp32 on this device."""
        for t in tensors:
            if t is None:
                continue
            if t.device != self.device or t.dtype != torch.float32 or not t.is_contiguous():
                raise ValueError(f"engine tensors must be contiguous fp32 on {self.device} "
                                 f"(got {t.dtype}, {t.device}, contiguous={t.is_contiguous()})")

    def _call(self, name, *args, work=None):
        if self.profile is None:
            _lib.check(getattr(self.lib, name)(*args), name)
            return
        if work is None and name == "fh_snake_aa_chunked":  # algorithmic bytes: fp32 in + fp32 / 16-bit out per element
            work = {"bytes": float(args[8] * args[9] * args[10]) * (8.0 if args[11] == 0 else 6.0)}
        if work is None and name == "fh_snake_aa_chunked_h":  # fp16 in + fp16 out
            work = {"bytes": float(args[8] * args[9] * args[10]) * 4.0, "tag": "fh_snake_aa_chunked"}
        if work is None and name == "fh_rmsnorm_f32":  # fp32 row in, fp32 / 16-bit row out  (args: ..., out_mode, rows, M, C, stream)
            work = {"bytes": float(args[6] * args[7]) * (8.0 if args[4] == 0 else 6.0)}
        self._profile_cool()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(torch.cuda.current_stream(self.device))
        _lib.check(getattr(self.lib, name)(*args), name)
        e1.record(torch.cuda.current_stream(self.device))
        self.profile.append((name, e0, e1, work or {}))

    def _profile_cool(self):
        """Profile mode only, FH_PROFILE_COOL_MS=x: drain the GPU and idle x ms before every launch, so each kernel is timed
        alone on a chip that is not at its power cap (tools/cool_vs_hot.py: is a kernel slow, or is the step power-limited?)."""
        if self._cool_ms > 0.0:
            import time
            torch.cuda.synchronize(self.device)
            time.sleep(self._cool_ms * 1e-3)

    def start_profile(self):
        """Brackets every kernel launch with CUDA events on the launching stream (bench.py roofline leg)."""
        self.profile = []

    def stop_profile(self):
        """-> {kernel: {"ms": total, "launches": n, "flops": f, "bytes": b}}"""
        torch.cuda.synchronize(self.device)
        agg = {}
        for name, e0, e1, work in self.profile or []:
            key = work.get("tag", name)
            d = agg.setdefault(key, {"ms": 0.0, "launches": 0, "flops": 0.0, "bytes": 0.0})
            d["ms"] += e0.elapsed_time(e1)
            d["launches"] += 1
            d["flops"] += work.get("flops", 0.0)
            d["bytes"] += work.get("bytes", 0.0)
        self.profile = None
        return agg

    # ------------------------------------------------------------------ weight preparation
    def _mk_f32(self, tconv: packing.TappedConv) -> _F32Weight:
        r = _F32Weight()
        r.w, r.off = packing.f32_conv_buffers(tconv, self.device)
        r.bias = None if tconv.bias is None else tconv.bias.to(self.device).float().contiguous()
        r.P, r.ntaps, r.cin, r.cout = tconv.P, tconv.ntaps, tconv.cin, tconv.cout
        return r

    def _pair_wins(self, cout: int, ntaps: int, P: int, residual: bool) -> bool:
        """Shapes on which the CTA-pair kernel beats the single-CTA kernel (B = 64 breakdowns of both in one gpurun call,
        profiles/r2_pair_vs_single.txt): 192 / 384 output channels with >= 7 taps gain 14-25 % (their weight stream per SM
        halves), the 96-channel k = 11 first convolutions 17 %; HBM-bound residual launches, k = 3 shapes, the upsamplers
        and the Linear layers lose 3-20 % to the two extra barrier hops per stage; 768 channels are at the tensor peak
        either way.  Decided per layer at load time because the packed weight layout differs."""
        if P != 1:
            return False
        if 192 <= cout <= 384 and ntaps >= 7:
            return True
        return cout == 96 and ntaps >= 11 and not residual

    def _mk_tc(self, tconv: packing.TappedConv, cin_pad=None, cout_pad=None, bn=None, split=False, two_cta=False) -> _TcWeight:
        r = _TcWeight()
        cin_alg = tconv.cin
        r.two_cta = bool(two_cta)
        if split:  # hi + lo activation operand: doubled input channels, duplicated weights
            cin_pad = cin_pad or packing.round_up(tconv.cin, 8)
            tconv = packing.split_input(tconv, cin_pad)
            cin_pad = 2 * cin_pad
        r.packed, r.cin_pad, r.cout_pad, r.bn = packing.pack_tc(tconv, self.device, cin_pad, cout_pad, bn, self.h16,
                                                                 two_cta=r.two_cta)
        r.bias = None if tconv.bias is None else packing.pad_vec(tconv.bias.to(self.device), r.cout_pad)
        r.off = tconv.off.copy()
        r.off_c = (C.c_int * r.off.size)(*[int(v) for v in r.off.flatten()])
        r.P, r.ntaps, r.cin, r.cout = tconv.P, tconv.ntaps, cin_alg, tconv.cout  # cin: algorithmic (FLOP accounting)
        return r

    def _prep_backbone(self):
        sd, b = self.sd, self.bcfg
        self.inner = b.ff_inner
        self.inner_pad = packing.round_up(self.inner, 16)
        if not self.tc:
            if b.architecture == "convnext":  # fp32 path: gamma * (W2 x + b2) folded once
                self.cn_f32 = [((sd[FH + f"convnext.{i}.pwconv2.weight"] * sd[FH + f"convnext.{i}.gamma"][:, None]).contiguous(),
                                (sd[FH + f"convnext.{i}.pwconv2.bias"] * sd[FH + f"convnext.{i}.gamma"]).contiguous())
                               for i in range(b.convnext_layers)]
            return
        L = {}
        L["to_embed"] = self._mk_tc(packing.linear_taps(sd[FH + "to_embed.weight"], sd[FH + "to_embed.bias"]))
        L["to_pred"] = self._mk_tc(packing.linear_taps(sd[FH + "to_pred.weight"], None))
        if b.architecture == "convnext":
            for i in range(b.convnext_layers):
                p = FH + f"convnext.{i}."
                L[f"pw1{i}"] = self._mk_tc(packing.linear_taps(sd[p + "pwconv1.weight"], sd[p + "pwconv1.bias"]))
                gm = sd[p + "gamma"]  # layer scale folded into the second pointwise conv: gamma * (W x + b)
                L[f"pw2{i}"] = self._mk_tc(packing.linear_taps(sd[p + "pwconv2.weight"] * gm[:, None], sd[p + "pwconv2.bias"] * gm))
            self.bb_tc = L
            return
        for l in range(b.depth):
            p = FH + f"transformer.layers.{l}."
            L[f"qkv{l}"] = self._mk_tc(packing.linear_taps(sd[p + "3.to_qkv.weight"], None))
            L[f"out{l}"] = self._mk_tc(packing.linear_taps(sd[p + "3.to_out.weight"], None))
            # FF in: interleave (x_i, gate_i) rows so that GEGLU is a column-pair epilogue; pad inner to x16
            w1, b1 = sd[p + "5.0.weight"], sd[p + "5.0.bias"]
            ip = self.inner_pad
            wi = torch.zeros(2 * ip, b.dim, device=w1.device)
            bi = torch.zeros(2 * ip, device=w1.device)
            wi[0:2 * self.inner:2] = w1[: self.inner]
            wi[1:2 * self.inner:2] = w1[self.inner:]
            bi[0:2 * self.inner:2] = b1[: self.inner]
            bi[1:2 * self.inner:2] = b1[self.inner:]
            L[f"ff1{l}"] = self._mk_tc(packing.linear_taps(wi, bi), bn=256)
            w2 = torch.zeros(b.dim, ip, device=w1.device)
            w2[:, : self.inner] = sd[p + "5.3.weight"]
            L[f"ff2{l}"] = self._mk_tc(packing.linear_taps(w2, sd[p + "5.3.bias"]))
            if p + "0.weight" in sd:  # U-Net skip combiner Linear(2 dim -> dim) as two accumulating GEMMs (no concat)
                ws = sd[p + "0.weight"]
                L[f"skipA{l}"] = self._mk_tc(packing.linear_taps(ws[:, : b.dim].contiguous(), sd[p + "0.bias"]))
                L[f"skipB{l}"] = self._mk_tc(packing.linear_taps((ws[:, b.dim:] * b.skip_connect_scale).contiguous(), None))
        self.bb_tc = L

    def _snake_params(self, prefix: str, cpad: int):
        sd, v = self.sd, self.vcfg
        alpha = sd[prefix + "act.alpha"].cpu()
        beta = sd[prefix + "act.beta"].cpu() if v.activation == "snakebeta" else alpha
        if v.snake_logscale:
            alpha, beta = torch.exp(alpha), torch.exp(beta)
        inv_b = 1.0 / (beta + 1e-9)
        a = packing.pad_vec(alpha, cpad, 1.0).to(self.device)
        ib = packing.pad_vec(inv_b, cpad, 0.0).to(self.device)
        filt_up = sd[prefix + "upsample.filter"].flatten()
        filt_dn = sd[prefix + "downsample.lowpass.filter"].flatten()
        if not torch.equal(filt_up, filt_dn):
            raise ValueError("up/down anti-alias filters differ; the snake kernels expect one 12-tap filter")
        return a, ib, filt_up.contiguous()

    def _prep_vocoder(self):
        sd, v = self.sd, self.vcfg
        mk = (lambda t, residual=False, **kw: self._mk_tc(t, split=self.split, two_cta=self._pair_wins(
            t.cout, t.ntaps, t.P, residual), **kw)) if self.tc else (lambda t, residual=False, **kw: self._mk_f32(t))
        pad = (lambda c: packing.round_up(c, 8)) if self.tc else (lambda c: c)  # whole 8-channel chunks
        self.cpad = pad
        V = {}
        C0 = v.upsample_initial_channel
        kw = dict(cin_pad=pad(v.num_mels), cout_pad=pad(C0)) if self.tc else {}
        V["conv_pre"] = mk(packing.conv1d_taps(sd[VOC + "conv_pre.weight"], sd[VOC + "conv_pre.bias"]), **kw)
        nk = v.num_kernels
        for s, (u, k) in enumerate(zip(v.upsample_rates, v.upsample_kernel_sizes)):
            cin, cout = C0 // (2 ** s), v.stage_channels(s)
            kw = dict(cin_pad=pad(cin), cout_pad=pad(cout)) if self.tc else {}
            V[f"up{s}"] = mk(packing.conv_transpose1d_taps(sd[VOC + f"ups.{s}.0.weight"], sd[VOC + f"ups.{s}.0.bias"], u),
                             **kw)
            for j, (kk, dil) in enumerate(zip(v.resblock_kernel_sizes, v.resblock_dilation_sizes)):
                p = VOC + f"resblocks.{s * nk + j}."
                kw = dict(cin_pad=pad(cout), cout_pad=pad(cout)) if self.tc else {}
                for i, d in enumerate(dil):
                    if v.resblock == "1":
                        V[f"r{s}.{j}.c1.{i}"] = mk(packing.conv1d_taps(sd[p + f"convs1.{i}.weight"],
                                                                       sd[p + f"convs1.{i}.bias"], d), **kw)
                        V[f"r{s}.{j}.c2.{i}"] = mk(packing.conv1d_taps(sd[p + f"convs2.{i}.weight"],
                                                                       sd[p + f"convs2.{i}.bias"], 1), residual=True, **kw)
                        V[f"r{s}.{j}.a1.{i}"] = self._snake_params(p + f"activations.{2 * i}.", pad(cout))
                        V[f"r{s}.{j}.a2.{i}"] = self._snake_params(p + f"activations.{2 * i + 1}.", pad(cout))
                    else:
                        V[f"r{s}.{j}.c1.{i}"] = mk(packing.conv1d_taps(sd[p + f"convs.{i}.weight"],
                                                                       sd[p + f"convs.{i}.bias"], d), residual=True, **kw)
                        V[f"r{s}.{j}.a1.{i}"] = self._snake_params(p + f"activations.{i}.", pad(cout))
        clast = v.stage_channels(v.num_stages - 1)
        V["post_act"] = self._snake_params(VOC + "activation_post.", pad(clast))
        wpost = torch.zeros(pad(clast), 7, device=self.device)
        wpost[:clast] = sd[VOC + "conv_post.weight"][0]
        V["post_w"] = wpost.contiguous()
        V["post_b"] = float(sd[VOC + "conv_post.bias"].item())
        self.voc = V

    # ------------------------------------------------------------------ stage: resample + normalise
    def resample_normalise(self, x: torch.Tensor, sr_in: int, sr_out: int = 48000, method: str = "scipy") -> torch.Tensor:
        """x [B, T_in] fp32 on device -> cond [B, T] = resample(x) / max|.|: `method='scipy'` is
        scipy.signal.resample_poly's filter (flowhighsr.py:68-69), `'soxr_hq'` the filter of the librosa branch
        (flowhighsr.py:74-80; tables.resample_plan_soxr_hq) -- same polyphase kernel, different taps."""
        return self.resample_normalise_parts([(x, sr_in)], sr_out, method)

    def resample_normalise_parts(self, parts: Sequence[Tuple[torch.Tensor, int]], sr_out: int = 48000,
                                 method: str = "scipy") -> torch.Tensor:
        """Clips of several input rates with one output length in one batch: parts [(x_r [B_r, T_r], sr_r)] ->
        cond [sum B_r, T_out], rows in part order, each row exactly what `resample_normalise` gives for it alone.  One
        resampler launch per part into its rows of the shared buffer (a 48 kHz part is copied there), then one
        normalisation launch for the whole batch."""
        for x, _ in parts:
            self._chk(x)
        if method not in ("scipy", "soxr_hq"):
            raise ValueError(f"unknown resampling method {method!r} (scipy|soxr_hq)")
        if not parts:
            raise ValueError("resample_normalise_parts needs at least one part")
        plans, T_out = [], None
        for x, sr_in in parts:
            plan = tables.resample_plan(sr_in, sr_out) if method == "scipy" else tables.resample_plan_soxr_hq(sr_in, sr_out)
            n = x.shape[1] if plan is None else tables.resample_out_len(x.shape[1], plan[1], plan[2])
            if T_out is not None and n != T_out:
                raise ValueError(f"parts resample to different lengths ({T_out} and {n} samples)")
            plans.append(plan)
            T_out = n
        B = sum(x.shape[0] for x, _ in parts)
        absmax = self.buf("rs_absmax", (B,), torch.int32)
        self._call("fh_fill_u32", absmax.data_ptr(), 0, B, self.stream)
        if len(parts) == 1 and plans[0] is None:  # 48 kHz in, one part: normalised straight from the input
            y = parts[0][0]
            self._call("fh_absmax_f32", y.data_ptr(), absmax.data_ptr(), B, T_out, self.stream)
        else:
            y = self.buf("rs_y", (B, T_out), zero=False)
            r0 = 0
            for (x, sr_in), plan in zip(parts, plans):
                B_r, T_in = x.shape
                if plan is None:
                    y[r0: r0 + B_r].copy_(x)
                    self._call("fh_absmax_f32", y[r0:].data_ptr(), absmax[r0:].data_ptr(), B_r, T_out, self.stream)
                else:
                    h, up, down, npp, npr = plan
                    key = (sr_in, sr_out, method)
                    if key not in self._resample_taps:
                        self._resample_taps[key] = torch.from_numpy(h).to(self.device)
                    hd = self._resample_taps[key]
                    self._call("fh_resample_poly_f32", x.data_ptr(), y[r0:].data_ptr(), hd.data_ptr(), absmax[r0:].data_ptr(),
                               B_r, T_in, T_out, hd.numel(), up, down, npp, npr, self.stream,
                               work={"bytes": 4.0 * B_r * (T_in + T_out), "flops": 2.0 * B_r * T_out * (hd.numel() // up + 1)})
                r0 += B_r
        cond = torch.empty((B, T_out), dtype=torch.float32, device=self.device)
        self._call("fh_scale_by_absmax_f32", y.data_ptr(), cond.data_ptr(), absmax.data_ptr(), 1.0, B, T_out, self.stream,
                   work={"bytes": 8.0 * B * T_out})
        return cond

    # ------------------------------------------------------------------ stage: log-mel
    def encode(self, audio: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """MelVoco.encode (melvoco.py:56-86): audio [B,T] -> log-mel [B,N,256]."""
        self._chk(audio, out)
        B, T = audio.shape
        if T < 785:
            raise ValueError("audio shorter than 785 samples cannot be reflect-padded by 784 (melvoco.py:74)")
        N = (T + 1568 - 2048) // 480 + 1
        mel = out if out is not None else torch.empty((B, N, 256), dtype=torch.float32, device=self.device)
        self._call("fh_stft_logmel_f32", audio.data_ptr(), mel.data_ptr(), self.window.data_ptr(), self.twiddle.data_ptr(),
                   self.mel_start.data_ptr(), self.mel_len.data_ptr(), self.mel_w.data_ptr(), self.mel_stride, B, T, N,
                   1 if self.precise_mel else 0, self.stream,
                   work={"bytes": 4.0 * B * (T + N * 256), "flops": B * N * (5.0 * 2048 * 11 + 2.0 * 2030)})
        return mel

    # ------------------------------------------------------------------ stage: backbone
    def _time_cond(self, t: float) -> dict:
        """time embedding + the 4 (gamma, beta) pairs for time t (flow.py:242, transformer.py:82-88).
        t only takes the values of the ODE grid, so results are cached per value."""
        key = float(np.float32(t))
        hit = self._time_cache.get(key)
        if hit is not None:
            self._time_cache.move_to_end(key)
            if self._touch_log is not None:
                self._touch_log[id(hit)] = hit
            return hit
        sd, b = self.sd, self.bcfg
        D = b.dim
        four = torch.empty(D, device=self.device)
        temb = torch.empty(D, device=self.device)
        self._call("fh_sincos_embed_f32", sd[FH + "sinu_pos_emb.0.weights"].data_ptr(), key, four.data_ptr(), D // 2,
                   self.stream)
        self._call("fh_gemv_f32", sd[FH + "sinu_pos_emb.1.weight"].data_ptr(), four.data_ptr(),
                   sd[FH + "sinu_pos_emb.1.bias"].data_ptr(), temb.data_ptr(), D, D, 1, self.stream)
        out = {}
        if b.architecture == "convnext":  # AdaLayerNorm scale(t), shift(t) of every block (convnext.py:86-88)
            for i in range(b.convnext_layers):
                for nm in ("scale", "shift"):
                    v = torch.empty(D, device=self.device)
                    self._call("fh_gemv_f32", sd[FH + f"convnext.{i}.norm.{nm}.weight"].data_ptr(), temb.data_ptr(),
                               sd[FH + f"convnext.{i}.norm.{nm}.bias"].data_ptr(), v.data_ptr(), D, D, 0, self.stream)
                    out[(i, nm)] = v
            self._time_cache[key] = out
            if self._touch_log is not None:
                self._touch_log[id(out)] = out
            return out
        for l in range(b.depth):
            for idx in (2, 4):
                p = FH + f"transformer.layers.{l}.{idx}."
                for nm in ("gamma", "beta"):
                    v = torch.empty(D, device=self.device)
                    self._call("fh_gemv_f32", sd[p + f"to_{nm}.weight"].data_ptr(), temb.data_ptr(),
                               sd[p + f"to_{nm}.bias"].data_ptr(), v.data_ptr(), D, D, 0, self.stream)
                    out[(l, idx, nm)] = v
        self._time_cache[key] = out
        if self._touch_log is not None:
            self._touch_log[id(out)] = out
        while len(self._time_cache) > 512:
            self._time_cache.popitem(last=False)
        return out

    def _tc_conv(self, rec: _TcWeight, a, a_batch, a_chunk, a_row0, out, out_strides, out_bf16, B, L, res=None,
                 res_strides=(0, 0, 0), res_bf16=0, alpha=1.0, beta=0.0, accumulate=0, geglu=0, act=0, acc_src=None):
        args = _lib.TcConvArgs()
        args.a, args.a_batch, args.a_chunk, args.a_row0 = _ptr(a), a_batch, a_chunk, a_row0
        args.w, args.bias = rec.packed.data_ptr(), _ptr(rec.bias)
        args.res, args.out = _ptr(res), out.data_ptr()
        args.out_batch, args.out_chunk, args.out_row = out_strides
        args.res_batch, args.res_chunk, args.res_row = res_strides
        args.out_is_16, args.res_is_16, args.fp16 = int(out_bf16), int(res_bf16), self.fp16
        args.alpha, args.beta_res, args.accumulate, args.geglu = alpha, beta, int(accumulate), int(geglu)
        args.act = int(act)
        args.two_cta = 1 if rec.two_cta else 0
        args.acc_src = _ptr(acc_src)
        args.B, args.L, args.Cin, args.Cout = B, L, rec.cin_pad, rec.cout_pad
        args.ntaps, args.P, args.tap_off, args.bn = rec.ntaps, rec.P, rec.off_c, rec.bn
        flops = 2.0 * B * L * rec.P * rec.ntaps * rec.cin * rec.cout
        esz_o = 2 if out_bf16 else 4
        nbytes = B * L * rec.cin * 2 + B * L * rec.P * rec.cout * (esz_o + ((4 if acc_src is not None else esz_o) if accumulate else 0))
        if res is not None:
            nbytes += B * L * rec.P * rec.cout * (2 if res_bf16 else 4)
        work = {"flops": flops, "bytes": float(nbytes),
                "tag": f"tc_conv[Cin{rec.cin},Cout{rec.cout},k{rec.ntaps}x{rec.P}"
                       f"{',res' if res is not None else ''}]"}
        self._launch_conv(args, work)

    def _launch_conv(self, args, work):
        if self.profile is None:
            _lib.check(self.lib.fh_tc_conv(C.byref(args), self.stream), "fh_tc_conv")
            return
        self._profile_cool()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(torch.cuda.current_stream(self.device))
        _lib.check(self.lib.fh_tc_conv(C.byref(args), self.stream), "fh_tc_conv")
        e1.record(torch.cuda.current_stream(self.device))
        self.profile.append(("fh_tc_conv", e0, e1, work))

    def _sgemm(self, A, lda, W, ldw, bias, res, ldr, beta, alpha, out, ldc, M, N, K):
        self._call("fh_sgemm_nt_f32", A.data_ptr(), lda, W.data_ptr() if isinstance(W, torch.Tensor) else W, ldw,
                   _ptr(bias), _ptr(res), ldr, beta, alpha, out.data_ptr(), ldc, M, N, K, self.stream)

    def vector_field_step(self, x: torch.Tensor, cond: torch.Tensor, t: float, base: torch.Tensor, coef: float,
                          out: torch.Tensor, cond_packed: bool = False):
        """out = base + coef * v(t, x | cond)   -- one NFE with the CFM update folded into the
        to_pred GEMM epilogue (flow.py:180-274 + torchdiffeq euler/midpoint step)."""
        self._chk(x, cond, base, out)
        sd, b = self.sd, self.bcfg
        B, N, Din = x.shape
        M, D, H, Dh = B * N, b.dim, b.heads, b.dim_head
        tcnd = self._time_cond(t)
        st = self.stream
        E = self.buf("bb_E", (M, D), zero=False)
        h = self.buf("bb_h", (M, D), zero=False)
        qkv = self.buf("bb_qkv", (M, 3 * D), zero=False)
        if self.tc:
            Mp = packing.round_up(M, 128) + 64
            xc = self.buf("bb_xc", (2 * Din // 8, Mp, 8), self.h16)
            act = self.buf("bb_act", (D // 8, Mp, 8), self.h16)
            g = self.buf("bb_g", (self.inner_pad // 8, Mp, 8), self.h16)
            cs = Mp * 8
            self._call("fh_to_chunked_16", x.data_ptr(), 0, 1, Din, xc.data_ptr(), 0, cs, 0, 1, Din, M, self.fp16, st)
            if not cond_packed:
                self._call("fh_to_chunked_16", cond.data_ptr(), 0, 1, Din, xc.data_ptr() + (Din // 8) * cs * 2, 0, cs,
                           0, 1, Din, M, self.fp16, st)
            L = self.bb_tc
            rm = lambda ld: (0, 8, ld)  # row-major fp32 output strides (batch, chunk, row)
            self._tc_conv(L["to_embed"], xc, 0, cs, 0, E, rm(D), 0, 1, M)
        else:
            We = sd[FH + "to_embed.weight"]
            self._sgemm(x, Din, We, 2 * Din, sd[FH + "to_embed.bias"], None, 0, 0.0, 1.0, E, D, M, D, Din)
            self._sgemm(cond, Din, We.data_ptr() + Din * 4, 2 * Din, None, E, D, 1.0, 1.0, E, D, M, D, Din)
        wc = sd[FH + "conv_embed.dw_conv1d.0.weight"]
        self._call("fh_dwconv_gelu_res_f32", E.data_ptr(), wc.data_ptr(), sd[FH + "conv_embed.dw_conv1d.0.bias"].data_ptr(),
                   h.data_ptr(), B, N, D, wc.shape[-1], st, work={"bytes": 8.0 * M * D, "flops": 2.0 * M * D * wc.shape[-1]})
        if b.architecture == "convnext":
            self._convnext_blocks(h, tcnd, B, N, M, D, act if self.tc else None, cs if self.tc else 0, Mp if self.tc else 0)
            fw, fb = sd[FH + "final_layer_norm.weight"], sd[FH + "final_layer_norm.bias"]
            if self.tc:
                self._call("fh_layernorm_f32", h.data_ptr(), fw.data_ptr(), fb.data_ptr(), act.data_ptr(), self.k16, Mp, M, D,
                           1e-6, st)
                self._tc_conv(L["to_pred"], act, 0, cs, 0, out, rm(Din), 0, 1, M, res=base, res_strides=rm(Din), alpha=coef,
                              beta=1.0)
            else:
                a = self.buf("bb_a", (M, D), zero=False)
                self._call("fh_layernorm_f32", h.data_ptr(), fw.data_ptr(), fb.data_ptr(), a.data_ptr(), 0, 0, M, D, 1e-6, st)
                self._sgemm(a, D, sd[FH + "to_pred.weight"], D, None, base, Din, 1.0, coef, out, Din, M, Din, D)
            return
        skips = []
        for l in range(b.depth):
            p = FH + f"transformer.layers.{l}."
            if p + "0.weight" in sd:
                # transformer.py:213-218: x = Linear(cat(x, skip * scale)) = W[:, :D] x + b + (scale W[:, D:]) skip
                sk = skips.pop()
                h2 = self.buf("bb_h2", (M, D), zero=False)
                if self.tc:
                    self._call("fh_to_chunked_16", h.data_ptr(), 0, 1, D, act.data_ptr(), 0, cs, 0, 1, D, M, self.fp16, st)
                    self._tc_conv(L[f"skipA{l}"], act, 0, cs, 0, h2, rm(D), 0, 1, M)
                    self._tc_conv(L[f"skipB{l}"], sk, 0, cs, 0, h, rm(D), 0, 1, M, res=h2, res_strides=rm(D), beta=1.0)
                else:
                    ws = sd[p + "0.weight"]
                    self._sgemm(h, D, ws, 2 * D, sd[p + "0.bias"], None, 0, 0.0, 1.0, h2, D, M, D, D)
                    self._sgemm(sk, D, ws.data_ptr() + D * 4, 2 * D, None, h2, D, 1.0, float(b.skip_connect_scale), h, D,
                                M, D, D)
            elif b.use_unet_skip_connection:
                if self.tc:
                    sk = self.buf(f"bb_skip{l}", (D // 8, Mp, 8), self.h16)
                    self._call("fh_to_chunked_16", h.data_ptr(), 0, 1, D, sk.data_ptr(), 0, cs, 0, 1, D, M, self.fp16, st)
                else:
                    sk = self.buf(f"bb_skip{l}", (M, D), zero=False)
                    self._call("fh_axpby_f32", h.data_ptr(), None, 1.0, 0.0, sk.data_ptr(), M * D, st)
                skips.append(sk)
            if self.tc:
                self._call("fh_rmsnorm_f32", h.data_ptr(), tcnd[(l, 2, "gamma")].data_ptr(), tcnd[(l, 2, "beta")].data_ptr(),
                           act.data_ptr(), self.k16, Mp, M, D, st)
                self._tc_conv(L[f"qkv{l}"], act, 0, cs, 0, qkv, rm(3 * D), 0, 1, M)
            else:
                a = self.buf("bb_a", (M, D), zero=False)
                self._call("fh_rmsnorm_f32", h.data_ptr(), tcnd[(l, 2, "gamma")].data_ptr(), tcnd[(l, 2, "beta")].data_ptr(),
                           a.data_ptr(), 0, 0, M, D, st)
                self._sgemm(a, D, sd[p + "3.to_qkv.weight"], D, None, None, 0, 0.0, 1.0, qkv, 3 * D, M, 3 * D, D)
            if self.tc:
                # tcgen05 attention: q / k / v^T written directly as the MMA operand images (attention_tc5.cu).  The
                # profile tags are the names bench.py's attention roofline reads.
                ops = [self.buf(f"bb_{nm}5", (int(self.lib.fh_attention_tc5_operand_elems(w, B, H, N)),), self.h16)
                       for w, nm in enumerate(("q", "k", "v"))]
                self._call("fh_qknorm_rope_tiles", qkv.data_ptr(), sd[p + "3.q_norm.gamma"].data_ptr(),
                           sd[p + "3.k_norm.gamma"].data_ptr(), sd[FH + "transformer.rotary_emb.inv_freq"].data_ptr(),
                           *[t_.data_ptr() for t_ in ops], B, N, H, Dh, float(b.qk_norm_scale), self.fp16, st,
                           work={"bytes": (12.0 + 10.0) * B * N * H * Dh, "tag": "fh_qknorm_rope_split"})
                # algorithmic: q k^T and p v, 2 N^2 Dh each per head; bytes: q (hi + lo), k (hi + lo), v in, out (all 16-bit)
                self._call("fh_attention_tc5", *[t_.data_ptr() for t_ in ops], act.data_ptr(), self.k16, Mp, B, H, N, Dh,
                           self.fp16, st, work={"flops": 4.0 * B * H * N * N * Dh, "bytes": 2.0 * 6 * B * H * N * Dh,
                                                "tag": "fh_attention_tc"})
                self._tc_conv(L[f"out{l}"], act, 0, cs, 0, h, rm(D), 0, 1, M, res=h, res_strides=rm(D), beta=1.0)
                self._call("fh_rmsnorm_f32", h.data_ptr(), tcnd[(l, 4, "gamma")].data_ptr(), tcnd[(l, 4, "beta")].data_ptr(),
                           act.data_ptr(), self.k16, Mp, M, D, st)
                self._tc_conv(L[f"ff1{l}"], act, 0, cs, 0, g, (0, cs, 8), 1, 1, M, geglu=1)
                self._tc_conv(L[f"ff2{l}"], g, 0, cs, 0, h, rm(D), 0, 1, M, res=h, res_strides=rm(D), beta=1.0)
            else:
                q, k, v = (self.buf(f"bb_{nm}", (B, H, N, Dh), zero=False) for nm in ("q", "k", "v"))
                self._call("fh_qknorm_rope_f32", qkv.data_ptr(), sd[p + "3.q_norm.gamma"].data_ptr(),
                           sd[p + "3.k_norm.gamma"].data_ptr(), sd[FH + "transformer.rotary_emb.inv_freq"].data_ptr(),
                           q.data_ptr(), k.data_ptr(), v.data_ptr(), B, N, H, Dh, st)
                o = self.buf("bb_o", (M, D), zero=False)
                self._call("fh_attention_f32", q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr(), B, H, N, Dh,
                           float(b.qk_norm_scale), st)
                self._sgemm(o, D, sd[p + "3.to_out.weight"], D, None, h, D, 1.0, 1.0, h, D, M, D, D)
                f = self.buf("bb_a", (M, D), zero=False)
                self._call("fh_rmsnorm_f32", h.data_ptr(), tcnd[(l, 4, "gamma")].data_ptr(), tcnd[(l, 4, "beta")].data_ptr(),
                           f.data_ptr(), 0, 0, M, D, st)
                u = self.buf("bb_u", (M, 2 * self.inner), zero=False)
                self._sgemm(f, D, sd[p + "5.0.weight"], D, sd[p + "5.0.bias"], None, 0, 0.0, 1.0, u, 2 * self.inner, M,
                            2 * self.inner, D)
                gg = self.buf("bb_gg", (M, self.inner), zero=False)
                self._call("fh_geglu_f32", u.data_ptr(), gg.data_ptr(), M, self.inner, st)
                self._sgemm(gg, self.inner, sd[p + "5.3.weight"], self.inner, sd[p + "5.3.bias"], h, D, 1.0, 1.0, h, D, M,
                            D, self.inner)
        gam = sd[FH + "transformer.final_norm.gamma"]
        if self.tc:
            self._call("fh_rmsnorm_f32", h.data_ptr(), gam.data_ptr(), None, act.data_ptr(), self.k16, Mp, M, D, st)
            self._tc_conv(L["to_pred"], act, 0, cs, 0, out, rm(Din), 0, 1, M, res=base, res_strides=rm(Din), alpha=coef,
                          beta=1.0)
        else:
            a = self.buf("bb_a", (M, D), zero=False)
            self._call("fh_rmsnorm_f32", h.data_ptr(), gam.data_ptr(), None, a.data_ptr(), 0, 0, M, D, st)
            self._sgemm(a, D, sd[FH + "to_pred.weight"], D, None, base, Din, 1.0, coef, out, Din, M, Din, D)

    def _convnext_blocks(self, h, tcnd, B, N, M, D, act, cs, Mp):
        """8 x ConvNeXtBlock (convnext.py:46-63): h += gamma * pwconv2(gelu(pwconv1(AdaLN(dwconv7(h); t)))), in place."""
        sd, b, st = self.sd, self.bcfg, self.stream
        I = D * b.convnext_mult
        y = self.buf("bb_cn_y", (M, D), zero=False)
        rm = lambda ld: (0, 8, ld)
        for i in range(b.convnext_layers):
            p = FH + f"convnext.{i}."
            self._call("fh_dwconv_f32", h.data_ptr(), sd[p + "dwconv.weight"].data_ptr(), sd[p + "dwconv.bias"].data_ptr(),
                       y.data_ptr(), B, N, D, 7, st)
            if self.tc:
                L = self.bb_tc
                g = self.buf("bb_cn_g", (I // 8, Mp, 8), self.h16)
                self._call("fh_layernorm_f32", y.data_ptr(), tcnd[(i, "scale")].data_ptr(), tcnd[(i, "shift")].data_ptr(),
                           act.data_ptr(), self.k16, Mp, M, D, 1e-6, st)
                self._tc_conv(L[f"pw1{i}"], act, 0, cs, 0, g, (0, cs, 8), 1, 1, M, act=1)
                self._tc_conv(L[f"pw2{i}"], g, 0, cs, 0, h, rm(D), 0, 1, M, res=h, res_strides=rm(D), beta=1.0)
            else:
                a = self.buf("bb_a", (M, D), zero=False)
                u = self.buf("bb_cn_u", (M, I), zero=False)
                self._call("fh_layernorm_f32", y.data_ptr(), tcnd[(i, "scale")].data_ptr(), tcnd[(i, "shift")].data_ptr(),
                           a.data_ptr(), 0, 0, M, D, 1e-6, st)
                self._sgemm(a, D, sd[p + "pwconv1.weight"], D, sd[p + "pwconv1.bias"], None, 0, 0.0, 1.0, u, I, M, I, D)
                self._call("fh_gelu_f32", u.data_ptr(), u.data_ptr(), M, I, st)
                w2, b2 = self.cn_f32[i]  # layer scale folded into pwconv2 at load time
                self._sgemm(u, I, w2, I, b2, h, D, 1.0, 1.0, h, D, M, D, I)

    def mel_cutoff_bins(self, cond_mel: torch.Tensor) -> torch.Tensor:
        """mel_cutoff_bins (cfm_superresolution.py:154-159): per-clip 99.95 % energy bin of exp(mel)."""
        self._chk(cond_mel)
        B, N, Fm = cond_mel.shape
        cut = torch.empty((B,), dtype=torch.int32, device=self.device)
        self._call("fh_mel_cutoff_f32", cond_mel.data_ptr(), cut.data_ptr(), B, N, Fm, 0.9995, self.stream)
        return cut

    def mel_splice(self, lo: torch.Tensor, hi: torch.Tensor, cut: torch.Tensor) -> torch.Tensor:
        """mel_replace_ops (cfm_superresolution.py:146-152): bins below the cutoff from `lo`, the rest from `hi`."""
        self._chk(lo, hi)
        B, N, Fm = lo.shape
        out = torch.empty_like(lo)
        self._call("fh_mel_splice_f32", lo.data_ptr(), hi.data_ptr(), cut.data_ptr(), out.data_ptr(), B, N, Fm, self.stream)
        return out

    def _field_update(self, x, cond, null, t, base, coef, out, cond_scale, packed):
        """out = base + coef * v(t, x), with classifier-free guidance when cond_scale != 1 (flow.py:165-178)."""
        if cond_scale == 1.0:
            self.vector_field_step(x, cond, t, base, coef, out, cond_packed=packed)
            return self.tc
        n = x.numel()
        zero = self.buf("cfg_zero", x.shape)
        vc = self.buf("cfg_vc", x.shape, zero=False)
        vn = self.buf("cfg_vn", x.shape, zero=False)
        self.vector_field_step(x, cond, t, zero, 1.0, vc, cond_packed=False)
        self.vector_field_step(x, null, t, zero, 1.0, vn, cond_packed=False)
        # null + (logits - null) * s
        self._call("fh_axpby_f32", vn.data_ptr(), vc.data_ptr(), 1.0 - cond_scale, cond_scale, vc.data_ptr(), n, self.stream)
        self._call("fh_axpby_f32", base.data_ptr(), vc.data_ptr(), 1.0, coef, out.data_ptr(), n, self.stream)
        return False

    def _odeint_adaptive(self, y0: torch.Tensor, cond_mel: torch.Tensor, null, cond_scale: float, t0: float, t1: float, *,
                         tableau, atol: float, rtol: float, max_steps: int = 10000) -> torch.Tensor:
        """y(t1) by an embedded 5(4) Runge-Kutta pair under an integral step-size controller: the `use_torchode=True`
        branch (cfm_superresolution.py:259-276: to.Tsit5 + to.IntegralController in to.AutoDiffAdjoint).  torchode gives
        every clip of a batch its own time, step size and accept / reject history; the clips are independent, so they
        are solved one after the other with a scalar time each (the time conditioning is one vector per launch).  Stage
        states, the solution and the error estimate are `fh_rk_lincomb_f32` launches, the controller's error ratio is
        `fh_rk_scaled_sumsq_f32` (fp64, fixed summation order) read back once per attempted step."""
        from . import rk
        B, N, Din = y0.shape
        n = N * Din
        ctl = rk.IntegralController(atol=float(atol), rtol=float(rtol), order=tableau.order)
        out = torch.empty_like(y0)
        K = self.buf("rk_k", (8, 1, N, Din), zero=False)   # k_0 .. k_6, slot 7 = scratch (error estimate / f1 - f0)
        ys = self.buf("rk_ys", (1, N, Din), zero=False)
        zero = self.buf("rk_zero", (1, N, Din))
        ssq = self.buf("rk_ssq", (1,), torch.float64, zero=False)
        nullb = None if null is None else null[:1]
        st = self.stream
        self.ode_stats = []

        def field(x, cond, t, slot):  # K[slot] = v(t, x)
            self._field_update(x, cond, nullb, float(np.float32(t)), zero, 1.0, K[slot], cond_scale, False)

        def lincomb(base, coefs, dst):
            arr = (C.c_float * len(coefs))(*[float(c) for c in coefs])
            self._call("fh_rk_lincomb_f32", _ptr(base), K.data_ptr(), n, len(coefs), arr, dst.data_ptr(), n, st)

        def norm(e, ya, yb):
            self._call("fh_rk_scaled_sumsq_f32", e.data_ptr(), ya.data_ptr(), _ptr(yb), ctl.atol, ctl.rtol, 1, n,
                       ssq.data_ptr(), st)
            return float(np.sqrt(ssq.item() / n))

        for b in range(B):
            y = out[b: b + 1]
            self._call("fh_axpby_f32", y0[b: b + 1].data_ptr(), None, 1.0, 0.0, y.data_ptr(), n, st)
            cond = cond_mel[b: b + 1]
            t, span = t0, t1 - t0
            field(y, cond, t, 0)
            nfe = 1
            # Hairer's initial step: d0 = |y0|, d1 = |f0|, d2 = |f(t0 + h0, y0 + h0 f0) - f0| / h0 in the scaled rms norm
            d0, d1 = norm(y, y, None), norm(K[0], y, None)
            h0 = ctl.initial_dt(d0, d1, span)
            lincomb(y, [h0], ys)
            field(ys, cond, t + h0, 1)
            nfe += 1
            lincomb(None, [-1.0, 1.0], K[7])
            dt = ctl.initial_dt_refine(h0, d1, norm(K[7], y, None) / h0, span)
            n_steps = n_acc = 0
            while t < t1:
                if n_steps >= max_steps:
                    raise RuntimeError(f"adaptive solve did not reach t_end in {max_steps} steps (clip {b}, t = {t})")
                dt = min(dt, t1 - t)
                last = dt >= t1 - t
                for s in range(1, 7):
                    lincomb(y, [dt * w for w in tableau.a[s]], ys)
                    field(ys, cond, t + tableau.c[s] * dt, s)
                    nfe += 1
                # ys now holds the 5th-order solution (FSAL: the last stage is evaluated at it)
                lincomb(None, [dt * w for w in tableau.e], K[7])
                ratio = norm(K[7], y, ys)
                n_steps += 1
                if ctl.accept(ratio):
                    t = t1 if last else t + dt
                    self._call("fh_axpby_f32", ys.data_ptr(), None, 1.0, 0.0, y.data_ptr(), n, st)
                    self._call("fh_axpby_f32", K[6].data_ptr(), None, 1.0, 0.0, K[0].data_ptr(), n, st)
                    n_acc += 1
                dt = ctl.next_dt(dt, ratio)
            self.ode_stats.append({"n_steps": n_steps, "n_accepted": n_acc, "n_f_evals": nfe})
        return out

    def _rk4_step(self, y, cond, null, t0, t1, cond_scale, packed):
        """One step of torchdiffeq's `rk4` (rk4_alt_step_func: the 3/8 rule, last stage at the grid point t1), y in place:
        k1 = f(t0, y), k2 = f(t0 + dt/3, y + dt k1/3), k3 = f(t0 + 2dt/3, y + dt (k2 - k1/3)), k4 = f(t1, y + dt (k1 - k2 + k3)),
        y += (k1 + 3 (k2 + k3) + k4) dt / 8.  Stage times in fp32 like the reference's fp32 grid; the last NFE writes
        y + dt (k1 + 3 k2 + 3 k3) / 8 + dt/8 k4 from its to_pred epilogue."""
        n = y.numel()
        K = self.buf("rk4_k", (3,) + tuple(y.shape), zero=False)
        ys = self.buf("rk4_ys", y.shape, zero=False)
        yb = self.buf("rk4_yb", y.shape, zero=False)
        zero = self.buf("rk4_zero", y.shape)
        st = self.stream
        t0, t1 = np.float32(t0), np.float32(t1)
        dt = np.float32(t1 - t0)
        third = float(dt) / 3.0

        def lincomb(coefs, dst):
            arr = (C.c_float * len(coefs))(*coefs)
            self._call("fh_rk_lincomb_f32", y.data_ptr(), K.data_ptr(), n, len(coefs), arr, dst.data_ptr(), n, st)

        packed = self._field_update(y, cond, null, float(t0), zero, 1.0, K[0], cond_scale, packed)
        lincomb([third], ys)
        packed = self._field_update(ys, cond, null, float(t0 + dt * np.float32(1.0 / 3.0)), zero, 1.0, K[1], cond_scale,
                                    packed)
        lincomb([-third, float(dt)], ys)
        packed = self._field_update(ys, cond, null, float(t0 + dt * np.float32(2.0 / 3.0)), zero, 1.0, K[2], cond_scale,
                                    packed)
        lincomb([float(dt), -float(dt), float(dt)], ys)
        lincomb([0.125 * float(dt), 0.375 * float(dt), 0.375 * float(dt)], yb)
        return self._field_update(ys, cond, null, float(t1), yb, 0.125 * float(dt), y, cond_scale, packed)

    def _odeint_dopri5(self, y0: torch.Tensor, cond_mel: torch.Tensor, null, cond_scale: float, t0: float, t1: float, *,
                       atol: float, rtol: float, joint: bool, max_steps: int = 10000) -> torch.Tensor:
        """y(t1) by torchdiffeq's `dopri5` (cfm_superresolution.py:243 with `torchdiffeq_ode_method='dopri5'`): Dormand-Prince
        stages with FSAL, Shampine's error estimate, torchdiffeq's controller (`rk.TorchdiffeqController`) and its quartic
        dense output at t1 from the last accepted step, which ends at or past t1 (the field is evaluated at t > 1 then).
        torchdiffeq solves whatever tensor it is given as ONE problem: one step sequence, the rms error norm over the
        whole tensor.  `joint=True` does that for the batch (`sample()` with B > 1); `joint=False` solves every clip on its
        own (`generate` is batch-1 in the reference, so the `generate*` paths see per-clip step sequences).  Times and
        controller arithmetic are fp64 on the host, the field gets fp32 times; one 8-byte read per attempted step."""
        B, N, Din = y0.shape
        inst = [(0, B)] if joint else [(b, b + 1) for b in range(B)]
        Bi = inst[0][1] - inst[0][0]
        n = Bi * N * Din
        tab = rk.DOPRI5
        ctl = rk.TorchdiffeqController(atol=float(atol), rtol=float(rtol))
        out = torch.empty_like(y0)
        K = self.buf("rk_k", (8, Bi, N, Din), zero=False)   # k_0 .. k_6, slot 7 = scratch (error estimate / f1 - f0)
        ys = self.buf("rk_ys", (Bi, N, Din), zero=False)
        zero = self.buf("rk_zero", (Bi, N, Din))
        ssq = self.buf("rk_ssq", (1,), torch.float64, zero=False)
        st = self.stream
        self.ode_stats = []
        f32 = np.float32

        def lincomb(base, coefs, dst):
            arr = (C.c_float * len(coefs))(*[float(c) for c in coefs])
            self._call("fh_rk_lincomb_f32", _ptr(base), K.data_ptr(), n, len(coefs), arr, dst.data_ptr(), n, st)

        def norm(e, ya, yb):
            self._call("fh_rk_scaled_sumsq_f32", e.data_ptr(), ya.data_ptr(), _ptr(yb), ctl.atol, ctl.rtol, 1, n,
                       ssq.data_ptr(), st)
            return float(np.sqrt(ssq.item() / n))

        for b0, b1 in inst:
            y = out[b0: b1]
            self._call("fh_axpby_f32", y0[b0: b1].data_ptr(), None, 1.0, 0.0, y.data_ptr(), n, st)
            cond = cond_mel[b0: b1]
            nullb = None if null is None else null[b0: b1]
            packed = False

            def field(x, t, slot):  # K[slot] = v(float32(t), x)
                nonlocal packed
                packed = self._field_update(x, cond, nullb, float(f32(t)), zero, 1.0, K[slot], cond_scale, packed)

            t = float(t0)
            field(y, t, 0)
            # Hairer's initial step: d0 = |y0|, d1 = |f0|, d2 = |f(t0 + h0, y0 + h0 f0) - f0| / h0 in the scaled rms norm
            d0, d1 = norm(y, y, None), norm(K[0], y, None)
            h0 = ctl.initial_dt(d0, d1)
            lincomb(y, [h0], ys)
            field(ys, t + h0, 1)
            lincomb(None, [-1.0, 1.0], K[7])
            dt = ctl.initial_dt_refine(h0, d1, norm(K[7], y, None) / h0)
            nfe, n_steps, n_acc = 2, 0, 0
            while t < t1:
                if n_steps >= max_steps:
                    raise RuntimeError(f"adaptive solve did not reach t_end in {max_steps} steps (clip {b0}, t = {t})")
                # torchdiffeq casts t0, dt and t0 + dt to the state's fp32 for the stages; stages with c = 1 sit at t0 + dt
                t_end = t + dt
                t32, dt32 = f32(t), f32(dt)
                for s in range(1, 7):
                    lincomb(y, [dt32 * f32(w) for w in tab.a[s]], ys)
                    field(ys, f32(t_end) if tab.c[s] == 1.0 else t32 + f32(tab.c[s]) * dt32, s)
                nfe += 6
                # ys now holds the 5th-order solution (FSAL: the last stage is evaluated at it)
                lincomb(None, [dt32 * f32(w) for w in rk.DPS_C_ERROR], K[7])
                ratio = norm(K[7], y, ys)
                n_steps += 1
                if ctl.accept(ratio):
                    n_acc += 1
                    if t_end >= t1:  # dense output at t1 from (y0, k_0 .. k_6) of this step
                        x = f32((t1 - t) / (t_end - t))
                        lincomb(y, rk.dopri5_dense_weights(float(x), float(dt32)), y)
                        break
                    t = t_end
                    self._call("fh_axpby_f32", ys.data_ptr(), None, 1.0, 0.0, y.data_ptr(), n, st)
                    self._call("fh_axpby_f32", K[6].data_ptr(), None, 1.0, 0.0, K[0].data_ptr(), n, st)
                dt = ctl.next_dt(dt, ratio)
            self.ode_stats.append({"n_steps": n_steps, "n_accepted": n_acc, "n_f_evals": nfe})
        return out

    def sample_mel(self, cond_mel: torch.Tensor, eps: torch.Tensor, *, steps: int, ode_method: str, cfm_method: str,
                   sigma: float, cond_scale: float = 1.0, mel_pp: bool = False, std_1: Optional[float] = None,
                   std_2: Optional[float] = None, adaptive: Optional[dict] = None, atol: float = 1e-5,
                   rtol: float = 1e-5, joint: bool = False) -> torch.Tensor:
        """CFM sampler (cfm_superresolution.py:162-284 up to `sampled`): prior + ODE solve (+ mel_pp).
        std_1 / std_2: the reference falls back to (1.0, sigma) unless BOTH are given (:180-183).
        ode_method: torchdiffeq's euler / midpoint / rk4 on the fixed grid linspace(0, 1, steps + 1), or its adaptive
        dopri5 under atol / rtol, solving the batch as one problem when `joint` (`sample()`) and clip by clip otherwise
        (`generate*`).  `adaptive` (use_torchode=True) takes priority over ode_method."""
        if std_1 is None or std_2 is None:
            std_1, std_2 = 1.0, float(sigma)
        rk.check_torchdiffeq_method(ode_method)
        self._chk(cond_mel, eps)
        B, N, Din = cond_mel.shape
        n = cond_mel.numel()
        y = torch.empty_like(cond_mel)
        cut = None
        if cfm_method == "basic_cfm":
            self._call("fh_axpby_f32", eps.data_ptr(), None, 1.0, 0.0, y.data_ptr(), n, self.stream)
        elif cfm_method in ("independent_cfm_adaptive", "independent_cfm_constant", "independent_cfm_mix"):
            # y0 = cond * std_1 + eps * std_2  (generate() always ends up with cond * 1 + eps * sigma: SURVEY F5)
            self._call("fh_axpby_f32", cond_mel.data_ptr(), eps.data_ptr(), float(std_1), float(std_2), y.data_ptr(), n,
                       self.stream)
            if cfm_method == "independent_cfm_mix":  # low bins from the adaptive prior, high bins pure noise (:232-237)
                cut = self.mel_cutoff_bins(cond_mel)
                y = self.mel_splice(y, eps, cut)
        else:
            raise ValueError(f"unknown cfm_method {cfm_method!r}")
        null = None
        if cond_scale != 1.0:
            null = torch.empty_like(cond_mel)
            self._call("fh_broadcast_row_f32", self.sd[FH + "null_cond"].data_ptr(), null.data_ptr(), B * N, Din, self.stream)
        tgrid = np.linspace(0.0, 1.0, steps + 1, dtype=np.float32)  # torch.linspace(0,1,steps+1) fp32
        ymid = torch.empty_like(y) if ode_method == "midpoint" else None
        packed = False
        if adaptive is not None:  # use_torchode=True (cfm_superresolution.py:259-276): only t_eval[0] / t_eval[-1] matter
            y = self._odeint_adaptive(y, cond_mel, null, cond_scale, float(tgrid[0]), float(tgrid[-1]), **adaptive)
            steps = 0
        elif ode_method == "dopri5":  # interior grid points are interpolated, never stepped to: only the end points matter
            y = self._odeint_dopri5(y, cond_mel, null, cond_scale, float(tgrid[0]), float(tgrid[-1]), atol=atol, rtol=rtol,
                                    joint=joint)
            steps = 0
        for i in range(steps):
            t0, t1 = tgrid[i], tgrid[i + 1]
            dt = np.float32(t1 - t0)
            if ode_method == "euler":
                packed = self._field_update(y, cond_mel, null, float(t0), y, float(dt), y, cond_scale, packed)
            elif ode_method == "rk4":
                packed = self._rk4_step(y, cond_mel, null, t0, t1, cond_scale, packed)
            else:
                half = np.float32(0.5) * dt
                packed = self._field_update(y, cond_mel, null, float(t0), y, float(half), ymid, cond_scale, packed)
                packed = self._field_update(ymid, cond_mel, null, float(np.float32(t0 + half)), y, float(dt), y,
                                            cond_scale, packed)
        if mel_pp:  # cfm_superresolution.py:278-279
            if cut is None:
                cut = self.mel_cutoff_bins(cond_mel)
            y = self.mel_splice(cond_mel, y, cut)
        return y

    # ------------------------------------------------------------------ stage: vocoder
    def vocoder(self, mel: torch.Tensor) -> torch.Tensor:
        """MelVoco.decode (melvoco.py:114-121): mel [B,N,256] -> wave [B, 480 N]."""
        self._chk(mel)
        if not self.tc:
            return self._vocoder_f32(mel)
        B, N, _ = mel.shape
        wave = torch.empty((B, N * self.vcfg.total_upsample), dtype=torch.float32, device=self.device)
        if self.split:
            self._vocoder_tc_split(mel, wave)
        else:
            self._vocoder_tc(mel, wave)
        return wave

    def _conv_f32(self, rec: _F32Weight, x, out, B, L, res=None, beta=0.0, alpha=1.0, accumulate=0):
        self._call("fh_conv1d_taps_f32", x.data_ptr(), rec.w.data_ptr(), _ptr(rec.bias), rec.off.data_ptr(), _ptr(res),
                   beta, alpha, int(accumulate), out.data_ptr(), B, rec.cin, rec.cout, L, rec.ntaps, rec.P, self.stream)

    def _vocoder_f32(self, mel: torch.Tensor) -> torch.Tensor:
        v, V, st = self.vcfg, self.voc, self.stream
        B, N, nm = mel.shape
        melT = self.buf("vf_melT", (B, nm, N), zero=False)
        self._call("fh_transpose_f32", mel.data_ptr(), melT.data_ptr(), B, N, nm, st)
        C0 = v.upsample_initial_channel
        x = self.buf("vf_pre", (B, C0, N), zero=False)
        self._conv_f32(V["conv_pre"], melT, x, B, N)
        L = N
        nk = v.num_kernels
        for s, u in enumerate(v.upsample_rates):
            ch = v.stage_channels(s)
            Lo = L * u
            X = self.buf(f"vf_X{s}", (B, ch, Lo), zero=False)
            self._conv_f32(V[f"up{s}"], x, X, B, L)
            L = Lo
            XJ = self.buf(f"vf_XJ{s}", (B, ch, L), zero=False)
            Y = self.buf(f"vf_Y{s}", (B, ch, L), zero=False)
            A = self.buf(f"vf_A{s}", (B, ch, L), zero=False)
            XS = self.buf(f"vf_XS{s}", (B, ch, L), zero=False)
            for j, dil in enumerate(v.resblock_dilation_sizes):
                cur = X
                for i in range(len(dil)):
                    last = i == len(dil) - 1
                    a1, ib1, f1 = V[f"r{s}.{j}.a1.{i}"]
                    self._call("fh_snake_aa_f32", cur.data_ptr(), A.data_ptr(), a1.data_ptr(), ib1.data_ptr(), f1.data_ptr(),
                               B, ch, L, st)
                    if v.resblock == "1":
                        self._conv_f32(V[f"r{s}.{j}.c1.{i}"], A, Y, B, L)
                        a2, ib2, f2 = V[f"r{s}.{j}.a2.{i}"]
                        self._call("fh_snake_aa_f32", Y.data_ptr(), A.data_ptr(), a2.data_ptr(), ib2.data_ptr(),
                                   f2.data_ptr(), B, ch, L, st)
                        conv = V[f"r{s}.{j}.c2.{i}"]
                    else:
                        conv = V[f"r{s}.{j}.c1.{i}"]
                    if last:  # fold the mean over resblocks (models.py:181-187) into the last epilogue
                        self._conv_f32(conv, A, XS, B, L, res=cur, beta=1.0 / nk, alpha=1.0 / nk, accumulate=j > 0)
                    else:
                        self._conv_f32(conv, A, XJ, B, L, res=cur, beta=1.0)
                        cur = XJ
            x = XS
        ch = v.stage_channels(v.num_stages - 1)
        a, ib, f = V["post_act"]
        A = self.buf("vf_Apost", (B, ch, L), zero=False)
        self._call("fh_snake_aa_f32", x.data_ptr(), A.data_ptr(), a.data_ptr(), ib.data_ptr(), f.data_ptr(), B, ch, L, st)
        wave = torch.empty((B, L), dtype=torch.float32, device=self.device)
        self._call("fh_convpost_tanh_f32", A.data_ptr(), V["post_w"].data_ptr(), V["post_b"], wave.data_ptr(), B, ch, L, st)
        return wave

    def _geom(self, C: int, L: int):
        """chunked geometry: rows per chunk, elements per chunk / batch."""
        Lp = HALO + packing.round_up(L, 128) + 64
        cs = Lp * 8
        return Lp, cs, (C // 8) * cs

    def _cbuf(self, name, B, C, L, dtype):
        Lp, cs, bs = self._geom(C, L)
        # Zero-initialised, and kernels only ever write rows [0, L): the halo AND the rows [L, Lp) stay zero forever --
        # the conv windows read them as the Conv1d zero padding.  Lp rounds L up to 128 rows, so the key carries the
        # EXACT L: a shorter clip that shares the 128-row bucket of a longer one must not see its stale tail rows.
        t = self.buf(f"{name}@{L}", (B * bs + 4096,), dtype)
        return t, cs, bs

    def _vocoder_tc(self, mel: torch.Tensor, wave: torch.Tensor):
        v, V, st = self.vcfg, self.voc, self.stream
        B, N, nm = mel.shape
        bf, f32 = self.h16, torch.float32
        melc, mcs, mbs = self._cbuf("vt_mel", B, nm, N, bf)
        self._call("fh_to_chunked_16", mel.data_ptr(), N * nm, 1, nm, melc.data_ptr(), mbs, mcs, HALO, B, nm, N, self.fp16, st)
        C0 = self.cpad(v.upsample_initial_channel)
        xb, xcs, xbs = self._cbuf("vt_pre", B, C0, N, bf)
        self._tc_conv(V["conv_pre"], melc, mbs, mcs, HALO, xb[HALO * 8:], (xbs, xcs, 8), 1, B, N)
        L = N
        nk = v.num_kernels
        a_in, a_cs, a_bs = xb, xcs, xbs
        # The AMP branches of a stage (one per resblock kernel size) are independent until their mean
        # (bigvgan/models.py:181-187).  Large batches run them back to back, accumulating the mean in place (measured
        # 2 ms per step cheaper than separate outputs + a sum pass).  Small batches do not fill 148 SMs: there each
        # branch writes its own pre-scaled output on its own stream (parallel CUDA-graph branches when captured) and
        # fh_sum_cast_f32 adds them.
        par = (self.branch_streams and B <= self.branch_streams_max_batch and nk > 1)
        main = torch.cuda.current_stream(self.device)
        if par:
            while len(self._branch_streams) < nk:
                self._branch_streams.append(torch.cuda.Stream(self.device))
        for s, u in enumerate(v.upsample_rates):
            ch = self.cpad(v.stage_channels(s))
            Lo = L * u
            X, cs, bs = self._cbuf(f"vt_X{s}", B, ch, Lo, f32)
            o = HALO * 8  # element offset of row t = 0
            strides = (bs, cs, 8)
            self._tc_conv(V[f"up{s}"], a_in, a_bs, a_cs, HALO, X[o:], strides, 0, B, L)
            L = Lo
            if par:
                ev_up = torch.cuda.Event()
                ev_up.record(main)
            outs = []
            # sequential branches: the last one adds the running mean (XS, fp32) and writes the stage output directly as
            # the 16-bit operand of the next upsampler -- no fp32 store of the mean, no separate cast pass
            fuse_cast = not par and nk > 1 and s + 1 < v.num_stages
            if fuse_cast:
                XBf, _, _ = self._cbuf(f"vt_XB{s}", B, ch, Lo, bf)
            for j, dil in enumerate(v.resblock_dilation_sizes):
                bt = f"_{j}" if par else ""  # parallel branches need their own scratch
                XJ, _, _ = self._cbuf(f"vt_XJ{s}{bt}", B, ch, Lo, f32)
                y16 = self.y16 and v.resblock == "1"  # the tensor between the two convs of a unit is fp16
                Y, _, _ = self._cbuf(f"vt_Y{s}{bt}" + ("h" if y16 else ""), B, ch, Lo, bf if y16 else f32)
                A = self._cbuf(f"vt_A{s}{bt}", B, ch, Lo, bf)[0]
                # parallel branches write their own output (summed below); sequential ones accumulate in place
                XSj, _, _ = self._cbuf(f"vt_XS{s}_{j}" if par else f"vt_XS{s}", B, ch, Lo, f32)
                outs.append(XSj)
                ctx = torch.cuda.stream(self._branch_streams[j]) if par else contextlib.nullcontext()
                if par:
                    self._branch_streams[j].wait_event(ev_up)
                with ctx:
                    st = self.stream
                    cur = X
                    for i in range(len(dil)):
                        last = i == len(dil) - 1
                        sn1 = V[f"r{s}.{j}.a1.{i}"]
                        self._call("fh_snake_aa_chunked", cur.data_ptr(), A.data_ptr(), sn1[0].data_ptr(), sn1[1].data_ptr(),
                                   sn1[2].data_ptr(), bs, cs, HALO, B, ch, L, self.k16, st)
                        if v.resblock == "1":
                            self._tc_conv(V[f"r{s}.{j}.c1.{i}"], A, bs, cs, HALO, Y[o:], strides, 1 if y16 else 0, B, L)
                            sn2 = V[f"r{s}.{j}.a2.{i}"]
                            if y16:
                                self._call("fh_snake_aa_chunked_h", Y.data_ptr(), A.data_ptr(), sn2[0].data_ptr(),
                                           sn2[1].data_ptr(), sn2[2].data_ptr(), bs, cs, HALO, B, ch, L, st)
                            else:
                                self._call("fh_snake_aa_chunked", Y.data_ptr(), A.data_ptr(), sn2[0].data_ptr(),
                                           sn2[1].data_ptr(), sn2[2].data_ptr(), bs, cs, HALO, B, ch, L, self.k16, st)
                            conv = V[f"r{s}.{j}.c2.{i}"]
                        else:
                            conv = V[f"r{s}.{j}.c1.{i}"]
                        if last and fuse_cast and j == nk - 1:
                            self._tc_conv(conv, A, bs, cs, HALO, XBf[o:], strides, 1, B, L, res=cur[o:], res_strides=strides,
                                          alpha=1.0 / nk, beta=1.0 / nk, accumulate=True, acc_src=XSj[o:])
                        elif last:
                            self._tc_conv(conv, A, bs, cs, HALO, XSj[o:], strides, 0, B, L, res=cur[o:], res_strides=strides,
                                          alpha=1.0 / nk, beta=1.0 / nk, accumulate=(j > 0 and not par))
                        else:
                            self._tc_conv(conv, A, bs, cs, HALO, XJ[o:], strides, 0, B, L, res=cur[o:], res_strides=strides,
                                          beta=1.0)
                            cur = XJ
                    if par:
                        done = torch.cuda.Event()
                        done.record(self._branch_streams[j])
                        main.wait_event(done)
            st = self.stream
            XS, _, _ = self._cbuf(f"vt_XS{s}", B, ch, Lo, f32)
            if par:
                if len(outs) > 4:
                    raise ValueError("at most 4 resblock kernel sizes per stage")
                ptrs = [t_.data_ptr() for t_ in outs] + [None] * (4 - len(outs))
            if s + 1 < v.num_stages:
                XB, _, _ = self._cbuf(f"vt_XB{s}", B, ch, L, bf)
                if par:
                    self._call("fh_sum_cast_f32", *ptrs, None, XB.data_ptr(), B * bs, self.fp16, st)
                elif not fuse_cast:
                    self._call("fh_cast_f32_16", XS.data_ptr(), XB.data_ptr(), B * bs, self.fp16, st)
                a_in, a_cs, a_bs = XB, cs, bs
            elif par:
                self._call("fh_sum_cast_f32", *ptrs, XS.data_ptr(), None, B * bs, self.fp16, st)
        self._post(XS, bs, cs, B, ch, L, wave)

    def _post(self, XS, bs, cs, B, ch, L, wave):
        """activation_post -> conv_post -> tanh (bigvgan/models.py:189-192) on the last stage's fp32 rows: one fused kernel
        (the activated tensor stays in shared memory); > 64 channels: two kernels through HBM."""
        V, st = self.voc, self.stream
        a, ib, f = V["post_act"]
        if ch <= 64:
            self._call("fh_snakepost_convpost_tanh", XS.data_ptr(), bs, cs, HALO, a.data_ptr(), ib.data_ptr(), f.data_ptr(),
                       V["post_w"].data_ptr(), V["post_b"], wave.data_ptr(), B, ch, L, st,
                       work={"bytes": 4.0 * B * L * (ch + 1), "flops": 2.0 * B * L * ch * (7 + 24)})
            return
        AP, _, _ = self._cbuf("vt_AP", B, ch, L, torch.float32)
        self._call("fh_snake_aa_chunked", XS.data_ptr(), AP.data_ptr(), a.data_ptr(), ib.data_ptr(), f.data_ptr(), bs, cs,
                   HALO, B, ch, L, 0, st)
        self._call("fh_convpost_tanh_chunked", AP.data_ptr(), bs, cs, HALO, V["post_w"].data_ptr(), V["post_b"],
                   wave.data_ptr(), B, ch, L, st, work={"bytes": 4.0 * B * L * (ch + 1), "flops": 2.0 * B * L * ch * 7})

    def _vocoder_tc_split(self, mel: torch.Tensor, wave: torch.Tensor):
        """precision "fp16x2": the same tcgen05 convolutions over hi + lo activation pairs.  Every MMA operand producer
        writes [round(x) | round(x - hi)] into a buffer of twice the channels (fh_to_chunked_16_split,
        fh_cast_f32_16_split, fh_snake_aa_chunked_split); the residual stream and the tensor between the two convolutions
        of an AMP unit stay fp32.  AMP branches run back to back, the mean accumulates in place."""
        v, V, st = self.vcfg, self.voc, self.stream
        B, N, nm = mel.shape
        h16, f32 = self.h16, torch.float32
        o = HALO * 8
        nmp = self.cpad(nm)
        melc, mcs, mbs2 = self._cbuf("vs_mel", B, 2 * nmp, N, h16)
        self._call("fh_to_chunked_16_split", mel.data_ptr(), N * nm, 1, nm, melc.data_ptr(), mbs2, mcs, HALO, B, nm, N, self.fp16, st)
        C0 = self.cpad(v.upsample_initial_channel)
        pre, pcs, pbs = self._cbuf("vs_pre32", B, C0, N, f32)
        self._tc_conv(V["conv_pre"], melc, mbs2, mcs, HALO, pre[o:], (pbs, pcs, 8), 0, B, N)
        a_in, a_cs, a_bs2 = self._cbuf("vs_pre16", B, 2 * C0, N, h16)
        self._call("fh_cast_f32_16_split", pre.data_ptr(), a_in.data_ptr(), pcs, C0 // 8, pbs, a_bs2, B, self.fp16, st)
        L, nk = N, v.num_kernels
        for s, u in enumerate(v.upsample_rates):
            ch = self.cpad(v.stage_channels(s))
            Lo = L * u
            X, cs, bs = self._cbuf(f"vs_X{s}", B, ch, Lo, f32)
            strides = (bs, cs, 8)
            self._tc_conv(V[f"up{s}"], a_in, a_bs2, a_cs, HALO, X[o:], strides, 0, B, L)
            L = Lo
            XJ, _, _ = self._cbuf(f"vs_XJ{s}", B, ch, L, f32)
            Y, _, _ = self._cbuf(f"vs_Y{s}", B, ch, L, f32)
            XS, _, _ = self._cbuf(f"vs_XS{s}", B, ch, L, f32)
            A, _, bs2 = self._cbuf(f"vs_A{s}", B, 2 * ch, L, h16)

            def snake(src, sn):
                self._call("fh_snake_aa_chunked_split", src.data_ptr(), A.data_ptr(), sn[0].data_ptr(), sn[1].data_ptr(),
                           sn[2].data_ptr(), bs, bs2, cs, HALO, B, ch, L, st,
                           work={"bytes": float(B) * ch * L * 8.0, "tag": "fh_snake_aa_chunked"})
            for j, dil in enumerate(v.resblock_dilation_sizes):
                cur = X
                for i in range(len(dil)):
                    last = i == len(dil) - 1
                    snake(cur, V[f"r{s}.{j}.a1.{i}"])
                    if v.resblock == "1":
                        self._tc_conv(V[f"r{s}.{j}.c1.{i}"], A, bs2, cs, HALO, Y[o:], strides, 0, B, L)
                        snake(Y, V[f"r{s}.{j}.a2.{i}"])
                        conv = V[f"r{s}.{j}.c2.{i}"]
                    else:
                        conv = V[f"r{s}.{j}.c1.{i}"]
                    if last:
                        self._tc_conv(conv, A, bs2, cs, HALO, XS[o:], strides, 0, B, L, res=cur[o:], res_strides=strides,
                                      alpha=1.0 / nk, beta=1.0 / nk, accumulate=j > 0)
                    else:
                        self._tc_conv(conv, A, bs2, cs, HALO, XJ[o:], strides, 0, B, L, res=cur[o:], res_strides=strides, beta=1.0)
                        cur = XJ
            if s + 1 < v.num_stages:
                a_in, a_cs, a_bs2 = self._cbuf(f"vs_XB{s}", B, 2 * ch, L, h16)
                self._call("fh_cast_f32_16_split", XS.data_ptr(), a_in.data_ptr(), cs, ch // 8, bs, a_bs2, B, self.fp16, st)
        self._post(XS, bs, cs, B, ch, L, wave)

    # ------------------------------------------------------------------ stage: post-processing
    def postprocess(self, pred: torch.Tensor, src: torch.Tensor) -> torch.Tensor:
        """PostProcessing.post_processing (postprocessing.py:18-41) per clip: pred [B,Tp], src [B,T] -> [B,T]."""
        self._chk(pred, src)
        B, T = src.shape
        Tp = pred.shape[1]
        NT, NTp = 1 + T // 480, 1 + Tp // 480
        nt = min(NT, NTp)
        st = self.stream
        if NT != NTp:
            raise ValueError("post-processing expects pred and src to span the same number of STFT frames")
        en = self.buf("pp_en", (B, 1025), zero=False)
        cut = self.buf("pp_cut", (B,), torch.int32)
        frames = self.buf("pp_fr", (B, nt, 2048), zero=False)
        # no spectrogram in HBM: energy pass over src (two frames per complex FFT), then per frame
        # FFT(pred + i src) -> split -> splice -> inverse FFT
        ws = self.buf("pp_ws", (self.lib.fh_pp_energy_ws_bytes(B, NT) // 8,), torch.float64, zero=False)
        self._call("fh_pp_src_energy_f32", src.data_ptr(), en.data_ptr(), ws.data_ptr(), self.window.data_ptr(),
                   self.twiddle.data_ptr(), B, T, NT, st, work={"bytes": 4.0 * B * T, "flops": B * NT * 0.5 * 5.0 * 2048 * 11})
        self._call("fh_pp_cutoff", en.data_ptr(), cut.data_ptr(), B, 0.99, st)
        # bytes: pred + src read once (algorithmic), windowed frames written (2048 per 480 new samples: the OLA input)
        self._call("fh_pp_fused_f32", pred.data_ptr(), src.data_ptr(), cut.data_ptr(), frames.data_ptr(),
                   self.window.data_ptr(), self.twiddle.data_ptr(), B, Tp, T, NT, st,
                   work={"bytes": 4.0 * B * (Tp + T) + 4.0 * B * NT * 2048, "flops": B * NT * 2.0 * 5.0 * 2048 * 11})
        y = self.buf("pp_y", (B, T), zero=False)
        absmax = self.buf("pp_absmax", (B,), torch.int32)
        self._call("fh_fill_u32", absmax.data_ptr(), 0, B, st)
        self._call("fh_pp_overlap_add_f32", frames.data_ptr(), y.data_ptr(), self.window.data_ptr(), absmax.data_ptr(), B,
                   nt, T, st, work={"bytes": 4.0 * B * (nt * 2048 + T)})
        out = torch.empty((B, T), dtype=torch.float32, device=self.device)
        self._call("fh_scale_by_absmax_f32", y.data_ptr(), out.data_ptr(), absmax.data_ptr(), 0.99, B, T, st,
                   work={"bytes": 8.0 * B * T})
        return out
