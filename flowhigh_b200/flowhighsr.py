"""Drop-in Python surface of the reference (`from flowhigh import FlowHighSR`).

Mirrors src/flowhigh/flowhighsr.py:21-149 (constructor knobs, `from_local`, `from_pretrained`,
`generate`, `set_cfm_method`), cfm_superresolution.py:95-131,162-175 (`sample`, `load`, `device`)
and the sub-module call surface used for per-stage checks (`model.flowhigh.audio_enc_dec.encode /
.decode`, `model.flowhigh.forward_with_cond_scale`, `model.postproc.post_processing`).  The classes
are `nn.Module`s only as parameter containers: `state_dict()` / `load_state_dict()` use the
reference's exact key layout (flowhigh_b200/weights.py), while every computation goes to the CUDA
kernels through flowhigh_b200.engine.Engine.  There is no CPU path.

Reference quirks kept on purpose (SURVEY.md F4, F5, H8): `from_local` builds the wrapper with the
constructor defaults (basic_cfm + midpoint + sigma 0); the adaptive/constant prior is
`cond + sigma * eps` whatever `std_2` is passed; `audio.max() > 1` triggers the /32768 scaling;
an unknown `cfm_method` passed to `sample` silently falls back to `self.cfm_method`.
"""
from __future__ import annotations

import collections
import json
import math
from pathlib import Path
from typing import Dict, List, Optional, Sequence, Union

import numpy as np
import torch
from torch import nn

from . import tables
from .config import BackboneConfig, CFM_METHODS, VocoderConfig
from .engine import Engine
from .weights import FH, VOC, fold_weight_norm, random_state_dict, state_dict_spec

REPO_ID = "ResembleAI/FlowHigh"


def _on_model_device(fn):
    """Runs a public entry point with the model's GPU as the current device: the kernels launch on
    `torch.cuda.current_stream(device)` and set per-device function attributes, so a model on cuda:1 must not be
    driven while cuda:0 is current."""
    import functools

    @functools.wraps(fn)
    def wrapper(self, *a, **k):
        owner = self if isinstance(self, FlowHighSR) else self._owner()
        dev = owner.device
        if dev.type != "cuda":
            return fn(self, *a, **k)  # _engine() raises the "no CPU path" error
        with torch.cuda.device(dev):
            return fn(self, *a, **k)
    return wrapper


class _Tree(nn.Module):
    """Parameter container that reproduces a dotted state_dict key layout."""

    def _put(self, path: List[str], tensor: torch.Tensor, as_buffer: bool):
        if len(path) == 1:
            if as_buffer:
                self.register_buffer(path[0], tensor)
            else:
                self.register_parameter(path[0], nn.Parameter(tensor, requires_grad=False))
            return
        child = self._modules.get(path[0])
        if child is None:
            child = _Tree()
            self.add_module(path[0], child)
        child._put(path[1:], tensor, as_buffer)


def _is_buffer(key: str) -> bool:
    return key.endswith(".filter") or key.endswith("inv_freq")


def group_by_output_length(lengths: Sequence[int], srs: Sequence[int], target_sr: int, method: str) -> Dict[tuple, List[int]]:
    """Clip indices of one batched call -> {(T_out, method): indices}.  Only the resampler depends on the input rate: every
    kernel behind it sees [B, T_out] rows, so clips of one output length (`tables.resample_out_len`; the input length
    when the input is already at `target_sr`) share one batch whatever their rate and input length.  Inside a group the
    clips of one (rate, input length) part are consecutive, because the resampler runs one launch per part over
    contiguous rows: parts in the order of their first clip, clips of a part in caller order."""
    groups: Dict[tuple, Dict[tuple, List[int]]] = {}
    for i, (n, s) in enumerate(zip(lengths, srs)):
        g = math.gcd(int(target_sr), int(s))
        T_out = tables.resample_out_len(int(n), int(target_sr) // g, int(s) // g)
        groups.setdefault((T_out, method), {}).setdefault((int(s), int(n)), []).append(i)
    return {key: [i for idxs in parts.values() for i in idxs] for key, parts in groups.items()}


class MelVoco(_Tree):
    """models/melvoco.py:16-46: log-mel encoder + BigVGAN decoder (parameters under `.vocoder`)."""

    def __init__(self, *, vocoder_config: Union[str, Path, VocoderConfig, None] = None, vocoder_path=None,
                 n_mels=256, sampling_rate=48000, f_max=24000, f_min=20, n_fft=2048, win_length=2048, hop_length=480,
                 vocoder="bigvgan", log=True):
        super().__init__()
        if vocoder != "bigvgan":
            raise ValueError("unsuitable vocoder name")
        if (n_mels, sampling_rate, f_max, f_min, n_fft, win_length, hop_length) != (256, 48000, 24000, 20, 2048, 2048, 480):
            raise ValueError("the B200 front-end kernels are specialised for the 48 kHz / 2048 / 480 / 256-mel setup")
        if isinstance(vocoder_config, VocoderConfig):
            self.vcfg = vocoder_config
        elif vocoder_config is None:
            self.vcfg = VocoderConfig.assumed_48k()
        else:
            self.vcfg = VocoderConfig.from_json(vocoder_config)
        self.vcfg.validate()
        self.n_mels, self.n_fft, self.hop_length, self.win_length = n_mels, n_fft, hop_length, win_length
        self.sampling_rate, self.f_min, self.f_max = sampling_rate, f_min, f_max
        self._pending_generator = None
        if vocoder_path is not None:  # init_vocoder.py:14-17: load ['generator'], fold weight norm
            ckpt = torch.load(str(vocoder_path), map_location="cpu")
            self._pending_generator = fold_weight_norm(ckpt["generator"])
        self._owner = None

    @property
    def latent_dim(self):
        return self.n_mels

    @_on_model_device
    def encode(self, audio: torch.Tensor) -> torch.Tensor:
        eng = self._owner()._engine()
        eng.new_call()
        eng.status_begin()
        return eng.encode(audio.to(self._owner().device, torch.float32).contiguous())

    @_on_model_device
    def decode(self, mel: torch.Tensor) -> torch.Tensor:
        eng = self._owner()._engine()
        eng.new_call()
        eng.status_begin()  # sub-boundary calls leave the check to the caller: model._check_status(engine)
        return eng.vocoder(mel.to(eng.device, torch.float32).contiguous()).unsqueeze(1)


class FLowHigh(_Tree):
    """models/flow.py:55-142: vector-field network, `architecture` = 'transformer' (the checkpoint) or 'convnext'."""

    def __init__(self, *, audio_enc_dec: Optional[MelVoco] = None, dim_in=None, dim=1024, depth=24, dim_head=64,
                 heads=16, ff_mult=4, conv_pos_embed_kernel_size=31, attn_qk_norm=True, architecture="transformer",
                 use_unet_skip_connection=False, skip_connect_scale=None, **unused):
        super().__init__()
        if architecture not in ("transformer", "convnext"):
            raise ValueError("Choose approriate architecture")  # flow.py:84-85
        if not attn_qk_norm:
            raise NotImplementedError("the attention kernels implement the qk-norm variant the checkpoint uses")
        if audio_enc_dec is None:
            raise ValueError("audio_enc_dec (MelVoco) is required")
        dim_in = dim if dim_in is None else dim_in
        # use_unet_skip_connection: the reference's Transformer option (transformer.py:123,150-153); the reference FLowHigh
        # never forwards it (SURVEY F3), so it is an extension of this constructor, OFF by default like the checkpoint.
        if depth % 2:
            raise ValueError("depth must be even (transformer.py:130)")
        self.bcfg = BackboneConfig(dim_in=dim_in, dim=dim, depth=depth, heads=heads, dim_head=dim_head,
                                   ff_mult=ff_mult, conv_pos_kernel=conv_pos_embed_kernel_size,
                                   architecture=architecture,
                                   use_unet_skip_connection=bool(use_unet_skip_connection),
                                   skip_connect_scale=2 ** -0.5 if skip_connect_scale is None else float(skip_connect_scale))
        if (dim_in, dim, heads, dim_head) != (256, 1024, 16, 64):
            raise ValueError("kernels are specialised for dim_in 256, dim 1024, 16 heads x 64")
        self.audio_enc_dec = audio_enc_dec
        self._owner = None

    @_on_model_device
    def forward_with_cond_scale(self, x, *, times, cond, cond_scale=1.0, cond_mask=None, self_attn_mask=None):
        """flow.py:165-178: returns the vector field v(times, x | cond)."""
        if cond_mask is not None or self_attn_mask is not None:
            # generate() / sample() never pass them (cfm_superresolution.py:196,209-210: self_attn_mask = None,
            # cond_mask = None); the attention kernels have no masked form, so a mask must not be silently dropped
            raise NotImplementedError("cond_mask / self_attn_mask are not supported by the B200 attention kernels")
        eng = self._owner()._engine()
        eng.new_call()
        eng.status_begin()
        x = x.to(eng.device, torch.float32).contiguous()
        cond = cond.to(eng.device, torch.float32).contiguous()
        zero = torch.zeros_like(x)
        out = torch.empty_like(x)
        null = None
        if cond_scale != 1.0:
            null = eng.sd["flowhigh.null_cond"].expand_as(cond).contiguous()
        eng._field_update(x, cond, null, float(times), zero, 1.0, out, float(cond_scale), False)
        return out

    forward = forward_with_cond_scale


class PostProcessing:
    """postprocessing.py:5-41."""

    def __init__(self, owner):
        self._owner = owner

    @_on_model_device
    def post_processing(self, pred: torch.Tensor, src: torch.Tensor, length: int) -> torch.Tensor:
        assert pred.dim() == 2 and src.dim() == 2
        if length != src.shape[-1]:
            raise ValueError("length must equal src.size(-1) (the only way the reference calls it)")
        eng = self._owner()._engine()
        eng.new_call()
        return eng.postprocess(pred.to(eng.device, torch.float32).contiguous(), src.to(eng.device, torch.float32).contiguous())


class FlowHighSR(nn.Module):
    def __init__(self, flowhigh: FLowHigh, sigma=0.0, ode_atol=1e-5, ode_rtol=1e-5, use_torchode=False,
                 cfm_method="basic_cfm", torchdiffeq_ode_method="midpoint", torchode_method_klass=None,
                 cond_drop_prob=0.0, upsampling_method="scipy", precision: str = "fp16"):
        super().__init__()
        self.sigma = sigma
        self.flowhigh = flowhigh
        self.cond_drop_prob = cond_drop_prob
        self.use_torchode = use_torchode
        # the reference passes a torchode class (default torchode.Tsit5, flowhighsr.py:31); a name works too
        from . import rk
        self.torchode_method_klass = torchode_method_klass
        self._tableau = rk.resolve(torchode_method_klass) if use_torchode else None
        self.cfm_method = cfm_method
        self.odeint_kwargs = dict(atol=ode_atol, rtol=ode_rtol, method=torchdiffeq_ode_method)
        self.upsampling_method = upsampling_method
        self.precision = precision
        self.cuda_graphs = True          # capture small-batch generate() pipelines into CUDA graphs
        self.cuda_graph_max_batch = 8
        # Graphs are keyed by the exact input shape.  A service rarely sees a length twice, so a shape is captured only
        # when it comes back (`cuda_graph_min_hits`-th sighting; the eager run costs a third of a capture), and at most
        # `cuda_graph_cache_size` graphs (with their static buffers and private pools) are kept, least recently used out.
        # generate_batch(out_host=...): groups of >= 2 x this many clips run as two sub-batches so that the D2H copy of the first
        # overlaps the second.  OFF by default: at 64 x 10 s the two 32-clip halves cost 6 ms more than the 4 ms of PCIe
        # time they hide (tools/e2e_ab.py: 313.3 vs 310.9 ms per step; resident 303.9) -- worth it only for slower links.
        self.overlap_min_batch = 1 << 30
        self.readback_chunk = 16  # generate_batch(out_host=...): post-processing + read-back in chunks of this many clips (0: off)
        self.cuda_graph_min_hits = 2
        self.cuda_graph_cache_size = 8
        self._graphs: "collections.OrderedDict[tuple, tuple]" = collections.OrderedDict()
        self._graph_seen: "collections.OrderedDict[tuple, int]" = collections.OrderedDict()
        self.overflow_check = "raise"    # 16-bit paths: "raise" FloatingPointError on a saturated / non-finite operand, or "off"
        self._eng: Optional[Engine] = None
        import weakref
        ref = weakref.ref(self)
        flowhigh._owner = ref
        flowhigh.audio_enc_dec._owner = ref
        self.postproc = PostProcessing(ref)
        # parameters: random init of the named architecture until a checkpoint is loaded
        vcfg, bcfg = flowhigh.audio_enc_dec.vcfg, flowhigh.bcfg
        init = random_state_dict(bcfg, vcfg, seed=0, vocoder_gain=0.7)
        pend = flowhigh.audio_enc_dec._pending_generator
        if pend is not None:
            for k, v in pend.items():
                init[VOC + k] = v.float()
        for key, t in init.items():
            path = key.split(".")
            assert path[0] == "flowhigh"
            flowhigh._put(path[1:], t.clone(), _is_buffer(key))

    # ------------------------------------------------------------------ nn.Module protocol
    @property
    def device(self):
        return next(self.parameters()).device

    def _apply(self, fn, *a, **k):
        self._drop_engine()
        return super()._apply(fn, *a, **k)

    def load_state_dict(self, state_dict, strict: bool = True, **kw):
        self._drop_engine()
        return super().load_state_dict(state_dict, strict=strict, **kw)

    def load(self, path, strict=True):
        path = Path(path)
        assert path.exists()
        pkg = torch.load(str(path), map_location="cpu")
        self.load_state_dict(pkg["model"], strict=strict)
        return pkg

    def _engine(self) -> Engine:
        if self._eng is None:
            dev = self.device
            if dev.type != "cuda":
                raise RuntimeError("FlowHighSR (B200) needs its parameters on a CUDA device: call .cuda() / .to('cuda')")
            self._eng = Engine(self.state_dict(), self.flowhigh.audio_enc_dec.vcfg, self.flowhigh.bcfg, device=dev,
                               precision=self.precision)
        return self._eng

    def set_precision(self, precision: str):
        self.precision = precision
        self._drop_engine()

    def _drop_engine(self):
        self._eng = None
        self._graphs = collections.OrderedDict()
        self._graph_seen = collections.OrderedDict()

    # ------------------------------------------------------------------ reference API
    def set_cfm_method(self, cfm_method):
        self.cfm_method = cfm_method

    def _adaptive(self) -> Optional[dict]:
        """cfm_superresolution.py:240,259-276: `use_torchode` swaps the fixed-grid torchdiffeq solve for the adaptive one
        (atol / rtol from `odeint_kwargs`, the 5(4) pair from `torchode_method_klass`); `time_steps` then only fixes the
        end points of `t_eval`.  The accept / reject loop is host-driven, so these calls are never graph-captured."""
        if not self.use_torchode:
            return None
        return dict(tableau=self._tableau, atol=float(self.odeint_kwargs["atol"]), rtol=float(self.odeint_kwargs["rtol"]))

    def _host_driven_ode(self) -> bool:
        """Adaptive solves (torchode, torchdiffeq's dopri5) decide every step on the host: never graph-captured."""
        return self.use_torchode or self.odeint_kwargs["method"] == "dopri5"

    def _ode(self, joint: bool) -> dict:
        """ODE arguments of `Engine.sample_mel`.  `joint`: torchdiffeq's adaptive dopri5 solves the batch it is given as
        one problem (`sample()` with B > 1); the `generate*` paths are per clip like the reference's batch-1 `generate`."""
        return dict(ode_method=self.odeint_kwargs["method"], atol=float(self.odeint_kwargs["atol"]),
                    rtol=float(self.odeint_kwargs["rtol"]), adaptive=self._adaptive(), joint=joint)

    def _staging(self, numel: int) -> torch.Tensor:
        """Page-locked flat fp32 staging buffer of the batched host path (the clips of a group one after the other), cached
        per size (a few entries, least recently used out).  The previous upload from it must have left the host before it
        is refilled."""
        if getattr(self, "_stage_event", None) is None:
            self._stage_event = torch.cuda.Event()
            self._stage_bufs = collections.OrderedDict()
        else:
            self._stage_event.synchronize()
        buf = self._stage_bufs.get(numel)
        if buf is None:
            buf = self._stage_bufs[numel] = torch.empty(numel, dtype=torch.float32).pin_memory()
            while len(self._stage_bufs) > 4:
                self._stage_bufs.popitem(last=False)
        else:
            self._stage_bufs.move_to_end(numel)
        return buf

    def _resample_method(self) -> str:
        """flowhighsr.py:66-80: 'scipy' = resample_poly, 'librosa' = librosa.resample(res_type='soxr_hq').  Anything else
        leaves `cond` undefined in the reference (NameError); here it is a ValueError."""
        if self.upsampling_method == "scipy":
            return "scipy"
        if self.upsampling_method == "librosa":
            return "soxr_hq"
        raise ValueError(f"upsampling_method must be 'scipy' or 'librosa', got {self.upsampling_method!r}")

    def _noise_like(self, cond_mel: torch.Tensor, eps: Optional[torch.Tensor]) -> torch.Tensor:
        if eps is not None:
            return eps.to(cond_mel.device, torch.float32).reshape(cond_mel.shape).contiguous()
        return torch.randn_like(cond_mel)  # same draw the reference makes (cfm_superresolution.py:220)

    @torch.inference_mode()
    @_on_model_device
    def sample(self, *, cond=None, cond_mask=None, time_steps=4, cond_scale=1.0, decode_to_audio=True, std_1=None,
               std_2=None, mel_pp=False, cfm_method=None, eps: Optional[torch.Tensor] = None):
        if cfm_method not in CFM_METHODS:
            cfm_method = self.cfm_method
        if cond_mask is not None:
            raise NotImplementedError("cond_mask is not supported (generate() never passes one)")
        # cfm_superresolution.py:180-183: BOTH fall back to (1.0, sigma) unless both are given (SURVEY F5)
        if std_1 is None or std_2 is None:
            std_1, std_2 = 1.0, float(self.sigma)
        eng = self._engine()
        eng.new_call()
        eng.status_begin()
        cond = cond.to(eng.device, torch.float32).contiguous()
        is_audio = cond.dim() == 2 or (cond.dim() == 3 and cond.shape[1] == 1)
        if is_audio:
            cond = eng.encode(cond.reshape(cond.shape[0], -1))
        mel = eng.sample_mel(cond, self._noise_like(cond, eps), steps=int(time_steps), cfm_method=cfm_method,
                             sigma=float(self.sigma), cond_scale=float(cond_scale), mel_pp=bool(mel_pp), std_1=float(std_1),
                             std_2=float(std_2), **self._ode(joint=True))
        if not decode_to_audio:
            return mel
        out = eng.vocoder(mel).unsqueeze(1)
        self._check_status(eng)
        return out

    @staticmethod
    def _clip_len(audio) -> int:
        shp = tuple(audio.shape) if hasattr(audio, "shape") else np.asarray(audio).shape
        if len(shp) == 2 and shp[0] == 1:
            return int(shp[1])
        if len(shp) != 1:  # the reference's squeeze(0) would silently keep [C, T] and fail later
            raise ValueError(f"generate() takes mono audio, [T] or [1, T]; got shape {shp}")
        return int(shp[0])

    def _prep_input(self, audio) -> np.ndarray:
        if isinstance(audio, torch.Tensor):
            audio = audio.detach().cpu().numpy()
        audio = np.asarray(audio)
        if audio.ndim == 2:
            if audio.shape[0] != 1:  # the reference's squeeze(0) would silently keep [C, T] and fail later
                raise ValueError(f"generate() takes mono audio, [T] or [1, T]; got shape {tuple(audio.shape)}")
            audio = audio[0]
        elif audio.ndim != 1:
            raise ValueError(f"generate() takes mono audio, [T] or [1, T]; got shape {tuple(audio.shape)}")
        if audio.max() > 1:  # flowhighsr.py:62-63 (any dtype)
            audio = audio / 32768.0
        return np.ascontiguousarray(audio, dtype=np.float32)

    @torch.no_grad()
    def generate(self, audio, sr: int, target_sampling_rate=48000, timestep=1, eps: Optional[torch.Tensor] = None):
        """flowhighsr.py:51-102: one clip in, `[1, T]` fp32 tensor on the model device out."""
        out = self.generate_batch([audio], sr, target_sampling_rate, timestep, eps=None if eps is None else [eps])
        return out[0]

    @torch.no_grad()
    @_on_model_device
    def generate_batch(self, audios: Sequence, sr: Union[int, Sequence[int]], target_sampling_rate=48000, timestep=1,
                       eps: Optional[Sequence[torch.Tensor]] = None, pinned: bool = False,
                       out_host: Optional[torch.Tensor] = None) -> List[torch.Tensor]:
        """Batched `generate`: every clip is processed exactly as the reference processes it alone
        (per-clip peak normalisation, attention, cutoff and output normalisation; SURVEY.md F8).
        Clips with the same OUTPUT length run as one batch through every kernel, whatever their input rates and input
        lengths (`group_by_output_length`): the resampler runs once per (rate, input length) part of the batch, everything
        behind it once for the whole batch.  Clips of different output lengths run as separate batches; the results come
        back in caller order either way.

        `out_host` (optional, page-locked `[n_clips, T]` fp32): every result is ALSO copied there, asynchronously, on a
        side stream; groups of >= 2 * `overlap_min_batch` clips (off by default, see __init__) run as two sub-batches so
        that the device -> host copy of the first overlaps the kernels of the second (the output of a 64 x 10 s batch is
        123 MB, ~5 ms of PCIe time).  The caller synchronises the device (or `self.copy_stream`) before reading `out_host`."""
        method = self._resample_method()
        eng = self._engine()
        eng.new_call()
        srs = [int(s) for s in ([sr] * len(audios) if isinstance(sr, int) else sr)]
        # grouping needs the lengths only; the per-clip preparation (int16 heuristic = a pass over the samples, fp32 copy)
        # runs sub-batch by sub-batch below, so the host work of sub-batch k + 1 hides behind the kernels of sub-batch k
        prepped: List[Optional[np.ndarray]] = [None] * len(audios)
        lens = [self._clip_len(a) for a in audios]
        groups = group_by_output_length(lens, srs, int(target_sampling_rate), method)
        if out_host is not None:
            if not (out_host.is_pinned() and out_host.dtype == torch.float32 and out_host.dim() == 2
                    and out_host.shape[0] >= len(audios) and out_host.is_contiguous()):
                raise ValueError("out_host must be a contiguous page-locked fp32 tensor [n_clips, T]")
            if getattr(self, "copy_stream", None) is None:
                self.copy_stream = torch.cuda.Stream(eng.device)
            # sub-batches: [(output length, method), clip indices]
            work = []
            for key, idxs in groups.items():
                if len(idxs) >= 2 * self.overlap_min_batch:
                    h = (len(idxs) + 1) // 2
                    work += [(key, idxs[:h]), (key, idxs[h:])]
                else:
                    work.append((key, idxs))
        else:
            work = list(groups.items())
        results: List[Optional[torch.Tensor]] = [None] * len(audios)
        flags = 0
        check = self.overflow_check != "off" and eng.tc
        main = torch.cuda.current_stream(eng.device)
        for gi, ((T_out, _), idxs) in enumerate(work):
            if check and gi > 0 and out_host is None:
                flags |= eng.status_read()  # one status word per engine: collect the previous group's before the next resets it
            graphed = self.cuda_graphs and len(idxs) <= self.cuda_graph_max_batch and not self._host_driven_ode()
            # Clips that already sit in page-locked fp32 memory go to the device directly, one asynchronous copy each: no
            # staging copy, and no pass over the samples for the int16 heuristic (flowhighsr.py:62-63) -- dividing by
            # 32768 is an exact power-of-two scaling that the peak normalisation behind the resampler cancels bit for bit
            # (asserted by test_generate_batch_direct_pinned_and_chunked_readback).
            direct = pinned and not graphed and all(self._is_direct(audios[i]) for i in idxs)
            e = None if eps is None else torch.cat([eps[i].reshape(1, -1, 256) for i in idxs])
            pinned_done = False
            # with out_host the status word is reset once and accumulates over all sub-batches (no host sync in between)
            reset = out_host is None or gi == 0
            # the clips' samples one after the other, in `idxs` order: part r is a [count_r, n_r] block of it
            parts = self._parts(idxs, srs, lens)
            offs = np.cumsum([0] + [lens[i] for i in idxs]).tolist()
            if direct:
                x = torch.empty(offs[-1], dtype=torch.float32, device=eng.device)
                for j, i in enumerate(idxs):
                    x[offs[j]: offs[j + 1]].copy_(audios[i].reshape(-1), non_blocking=True)
                host = None
            else:
                for i in idxs:
                    prepped[i] = self._prep_input(audios[i])
                if pinned:  # one copy per clip into a cached page-locked staging buffer (no np.stack, no fresh cudaHostAlloc)
                    host = self._staging(offs[-1])
                    view = host.numpy()
                    for j, i in enumerate(idxs):
                        view[offs[j]: offs[j + 1]] = prepped[i]
                else:
                    host = torch.from_numpy(np.concatenate([prepped[i] for i in idxs]))

            def read_back(first, chunk):  # results of clips idxs[first : first + len(chunk)] -> out_host, on the copy stream
                if chunk.shape[1] > out_host.shape[1]:
                    raise ValueError(f"out_host rows hold {out_host.shape[1]} samples, a result has {chunk.shape[1]}")
                done = torch.cuda.Event()
                done.record(main)
                self.copy_stream.wait_event(done)
                sub = idxs[first: first + chunk.shape[0]]
                with torch.cuda.stream(self.copy_stream):
                    run0 = 0  # consecutive clip indices go out as one copy
                    while run0 < len(sub):
                        run1 = run0 + 1
                        while run1 < len(sub) and sub[run1] == sub[run1 - 1] + 1:
                            run1 += 1
                        out_host[sub[run0]: sub[run0] + (run1 - run0), : chunk.shape[1]].copy_(chunk[run0:run1], non_blocking=True)
                        run0 = run1
                chunk.record_stream(self.copy_stream)

            chunked = False
            if graphed and reset:
                outs = [self._run_group_graphed(eng, host, parts, T_out, int(target_sampling_rate), int(timestep), e)]
            else:
                if not direct:
                    x = host.to(eng.device, non_blocking=True)
                    if pinned:
                        self._stage_event.record(main)
                # large batches with a host destination: post-processing in chunks of `readback_chunk` clips, so that the
                # device -> host copy of a chunk overlaps the post-processing of the next (only the last chunk's copy is exposed)
                chunked = out_host is not None and self.readback_chunk and len(idxs) >= 2 * self.readback_chunk
                outs = self._run_group(eng, self._split(x, parts), int(target_sampling_rate), int(timestep),
                                       None if e is None else e.to(eng.device), reset_status=reset,
                                       pp_chunk=self.readback_chunk if chunked else 0, on_chunk=read_back if chunked else None)
                if not chunked:
                    outs = [outs]
                pinned_done = True
            if pinned and not pinned_done:  # graph path: the staging buffer is read by the copy in front of the replay
                self._stage_event.record(main)
            j0 = 0
            for chunk in outs:
                for j in range(chunk.shape[0]):
                    results[idxs[j0 + j]] = chunk[j: j + 1]
                if out_host is not None and not chunked:
                    read_back(j0, chunk)
                j0 += chunk.shape[0]
        if check:
            self._check_status(eng, flags | eng.status_read())
        return results  # type: ignore[return-value]

    @staticmethod
    def _parts(idxs: Sequence[int], srs: Sequence[int], lens: Sequence[int]) -> List[tuple]:
        """(rate, input length, count) of every run of consecutive clips of one rate and length in `idxs`."""
        parts: List[list] = []
        for i in idxs:
            if parts and parts[-1][:2] == [srs[i], lens[i]]:
                parts[-1][2] += 1
            else:
                parts.append([srs[i], lens[i], 1])
        return [tuple(p) for p in parts]

    @staticmethod
    def _split(x: torch.Tensor, parts: Sequence[tuple]) -> List[tuple]:
        """Flat device samples of a group -> [(x_r [count, n] view, rate)] per part."""
        out, o = [], 0
        for s, n, c in parts:
            out.append((x[o: o + c * n].view(c, n), s))
            o += c * n
        return out

    def _run_group(self, eng, parts, target_sr, timestep, eps_dev, reset_status: bool = True, pp_chunk: int = 0, on_chunk=None):
        """resample -> log-mel -> CFM -> vocoder -> post-processing for one batch of clips of one output length, given as
        parts [(x_r [count, n] on the device, rate)].
        `pp_chunk` > 0: the post-processing (per clip anyway) runs in chunks of that many clips, `on_chunk(first, out)` is
        called after each (the caller starts its device -> host copy there), and the list of chunk results is returned."""
        if reset_status:
            eng.status_begin()
        cond = eng.resample_normalise_parts(parts, target_sr, method=self._resample_method())
        cond_mel = eng.encode(cond)
        mel = eng.sample_mel(cond_mel, self._noise_like(cond_mel, eps_dev), steps=timestep, cfm_method=self.cfm_method,
                             sigma=float(self.sigma), **self._ode(joint=False))
        wave = eng.vocoder(mel)
        if pp_chunk <= 0:
            out = eng.postprocess(wave, cond)
            eng.status_end()
            return out
        outs = []
        for a in range(0, wave.shape[0], pp_chunk):
            o = eng.postprocess(wave[a: a + pp_chunk], cond[a: a + pp_chunk])
            if a + pp_chunk >= wave.shape[0]:
                eng.status_end()
            if on_chunk is not None:
                on_chunk(a, o)
            outs.append(o)
        return outs

    @staticmethod
    def _is_direct(a) -> bool:
        return (isinstance(a, torch.Tensor) and a.dtype == torch.float32 and a.device.type == "cpu" and a.is_pinned()
                and a.is_contiguous() and (a.dim() == 1 or (a.dim() == 2 and a.shape[0] == 1)))

    def _check_status(self, eng, flags: int = None):
        """16-bit paths: raises when a tensor-core operand left the fp16 range (saturated at +-65504) or was inf / NaN --
        the device-side replacement of the reference's per-NFE NaN prints (models/flow.py:256-267).  One stream
        synchronisation per generate() call; `overflow_check = "off"` skips it."""
        if self.overflow_check == "off" or not eng.tc:
            return
        if flags is None:
            eng.status_end()
            flags = eng.status_read()
        if flags:
            raise FloatingPointError(
                f"flowhigh_b200: a {eng.precision} tensor-core operand overflowed or was not finite (status {flags:#x}); "
                "the result is not trustworthy -- use precision='bf16' (fp32 range) or 'fp32' for these weights / inputs")

    def _run_group_graphed(self, eng, host, parts, T, target_sr, timestep, eps_host):
        """Small batches are launch-bound (~300 kernel launches per clip): the whole per-shape pipeline is captured
        into a CUDA graph (static input / noise / output buffers) and replayed.  `host` holds the group's samples flat,
        `parts` its ordered (rate, input length, count) parts, `T` its output length; a shape is that tuple of parts.
        A shape is captured when it is seen for the `cuda_graph_min_hits`-th time; the cache holds
        `cuda_graph_cache_size` graphs, least recently used out (each entry owns its static buffers, its private pool and
        references to the engine buffers it replays into)."""
        B = sum(c for _, _, c in parts)
        key = (tuple(parts), target_sr, timestep, self.odeint_kwargs["method"], self.cfm_method, float(self.sigma),
               self.upsampling_method)
        ent = self._graphs.get(key)
        if ent is None:
            seen = self._graph_seen.get(key, 0) + 1
            self._graph_seen[key] = seen
            self._graph_seen.move_to_end(key)
            while len(self._graph_seen) > 64 * max(1, self.cuda_graph_cache_size):
                self._graph_seen.popitem(last=False)
            if seen < self.cuda_graph_min_hits:
                x = host.to(eng.device, non_blocking=True)
                return self._run_group(eng, self._split(x, parts), target_sr, timestep,
                                       None if eps_host is None else eps_host.to(eng.device))
            x_static = torch.zeros(host.shape, dtype=torch.float32, device=eng.device)
            x_static.copy_(host)
            eps_static = torch.randn((B, T // 480, 256), dtype=torch.float32, device=eng.device)
            parts_static = self._split(x_static, parts)
            eng._touch_log = {}
            try:
                side = torch.cuda.Stream(eng.device)
                side.wait_stream(torch.cuda.current_stream(eng.device))
                with torch.cuda.stream(side):
                    for _ in range(2):  # allocate persistent buffers, time-conditioning cache, function attributes
                        self._run_group(eng, parts_static, target_sr, timestep, eps_static)
                torch.cuda.current_stream(eng.device).wait_stream(side)
                torch.cuda.synchronize(eng.device)
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    out_static = self._run_group(eng, parts_static, target_sr, timestep, eps_static)
                keep = list(eng._touch_log.values())
            finally:
                eng._touch_log = None
            ent = self._graphs[key] = (graph, x_static, eps_static, out_static, keep)
            while len(self._graphs) > max(1, self.cuda_graph_cache_size):
                self._graphs.popitem(last=False)
        else:
            self._graphs.move_to_end(key)
        graph, x_static, eps_static, out_static, _keep = ent
        x_static.copy_(host, non_blocking=True)
        if eps_host is not None:
            eps_static.copy_(eps_host.reshape(eps_static.shape), non_blocking=True)
        else:
            eps_static.normal_()
        graph.replay()
        return out_static.clone()

    @torch.no_grad()
    @_on_model_device
    def generate_long(self, audio, sr: int, target_sampling_rate=48000, timestep=1, chunk_seconds: float = 10.0,
                      overlap_seconds: float = 0.5, eps: Optional[torch.Tensor] = None, max_batch: int = 64,
                      group=None, distributed: Optional[bool] = None):
        """Long-form generation by overlapped chunking + overlap-add (SURVEY.md 8e; not in the reference,
        whose dense fp32 attention cannot hold a 10-minute clip).  The input is resampled and peak-normalised
        ONCE (global scalar), cut into uniform chunks in the 48 kHz domain, every chunk runs log-mel -> CFM ->
        vocoder as an independent clip, the vocoder outputs are cross-faded, and the STFT-domain
        post-processing (global cutoff bin, global output normalisation) runs once over the stitched signal.
        `eps` (optional) is [K, frames, 256].

        Multi-GPU (torch.distributed initialised, one process per GPU, every rank calls this with the same input):
        rank r runs a contiguous block of the K chunks, ONE all_gather_into_tensor (ncclAllGather) puts all chunk
        waveforms on every rank, and every rank stitches + post-processes (identical results, no second collective).
        Per-chunk results do not depend on the batch they ran in, so the output is bit-identical to the 1-GPU call."""
        import torch.distributed as dist
        from . import sharding
        eng = self._engine()
        eng.new_call()
        eng.status_begin()
        if distributed is None:
            distributed = dist.is_available() and dist.is_initialized()
        world = dist.get_world_size(group) if distributed else 1
        rank = dist.get_rank(group) if distributed else 0
        x = torch.from_numpy(self._prep_input(audio))[None].to(eng.device)
        cond = eng.resample_normalise(x, int(sr), target_sampling_rate, method=self._resample_method())  # [1, T]  (every rank: 0.1 % of the work)
        T = cond.shape[1]
        clen = int(round(chunk_seconds * 48000)) // 480 * 480
        ov = int(round(overlap_seconds * 48000)) // 480 * 480
        if T <= clen:
            return self.generate(audio, sr, target_sampling_rate, timestep, eps=None if eps is None else eps[0])
        step = clen - ov
        K = -(-(T - clen) // step) + 1
        Tpad = (K - 1) * step + clen
        padded = torch.zeros((1, Tpad), dtype=torch.float32, device=eng.device)
        padded[:, :T] = cond
        k0, k1, per = sharding.block_range(K, world, rank)
        chunks = padded.unfold(1, clen, step)[0][k0:k1].contiguous()  # [K_local, clen] (overlapped spans, copied once)
        waves = torch.empty((k1 - k0, clen), dtype=torch.float32, device=eng.device)
        if eps is None:  # the same noise on every rank: rank 0's seed (an 8-byte broadcast), all K chunks drawn everywhere
            seed = torch.randint(0, 2 ** 31 - 1, (1,), dtype=torch.int64, device=eng.device)
            if world > 1:
                dist.broadcast(seed, 0, group=group)
            g = torch.Generator(device=eng.device)
            g.manual_seed(int(seed.item()))
            eps = torch.randn((K, clen // 480, 256), dtype=torch.float32, device=eng.device, generator=g)
        for b0 in range(0, k1 - k0, max_batch):
            c = chunks[b0: b0 + max_batch]
            mel_c = eng.encode(c)
            e = eps[k0 + b0: k0 + b0 + c.shape[0]]
            mel = eng.sample_mel(mel_c, self._noise_like(mel_c, e), steps=int(timestep), cfm_method=self.cfm_method,
                                 sigma=float(self.sigma), **self._ode(joint=False))
            waves[b0: b0 + c.shape[0]] = eng.vocoder(mel)
        if world > 1:
            waves = sharding.gather_blocks(waves, per, K, group)  # the only collective of the path
        Tv = T // 480 * 480  # the vocoder emits whole frames (pred is shorter than src when T % 480 != 0)
        stitched = torch.empty((1, Tv), dtype=torch.float32, device=eng.device)
        eng._call("fh_ola_crossfade_f32", waves.data_ptr(), stitched.data_ptr(), K, clen, step, Tv, eng.stream)
        out = eng.postprocess(stitched, cond)
        self._check_status(eng)
        return out

    @torch.no_grad()
    @_on_model_device
    def generate_sharded(self, audios: Sequence, sr: Union[int, Sequence[int]], target_sampling_rate=48000, timestep=1,
                         eps: Optional[Sequence[torch.Tensor]] = None, max_batch: int = 64, group=None, gather: bool = True):
        """A list of clips (mixed input rates allowed, equal OUTPUT length) over the GPUs of one box: every rank calls
        this with the same list, `sharding.assign_clips` gives rank r its clips, they run through `generate_batch` in
        batches of <= max_batch per output-length group (clips of different input rates share a batch), and -- when
        `gather` -- ONE all_gather_into_tensor puts the [n_clips, T] fp32 result on every rank in clip order.  No
        collective on the data path itself."""
        import torch.distributed as dist
        from . import sharding
        distributed = dist.is_available() and dist.is_initialized()
        world = dist.get_world_size(group) if distributed else 1
        rank = dist.get_rank(group) if distributed else 0
        srs = [sr] * len(audios) if isinstance(sr, int) else list(sr)
        out_len = [-(-int(np.asarray(a).shape[-1]) * int(target_sampling_rate) // int(s)) for a, s in zip(audios, srs)]
        parts = sharding.assign_clips(out_len, world)
        mine = parts[rank]
        results: List[Optional[torch.Tensor]] = [None] * len(mine)
        groups = group_by_output_length([self._clip_len(audios[i]) for i in mine], [int(srs[i]) for i in mine],
                                        int(target_sampling_rate), self._resample_method())
        for js in groups.values():
            for b0 in range(0, len(js), max_batch):
                sel = js[b0: b0 + max_batch]
                outs = self.generate_batch([audios[mine[j]] for j in sel], [int(srs[mine[j]]) for j in sel],
                                           target_sampling_rate, timestep,
                                           eps=None if eps is None else [eps[mine[j]] for j in sel], pinned=True)
                for j, o in zip(sel, outs):
                    results[j] = o
        if not gather:
            return {i: results[j] for j, i in enumerate(mine)}
        if len(set(out_len)) > 1:
            raise ValueError("generate_sharded(gather=True) needs clips of one output length (use gather=False)")
        T = out_len[0] if out_len else 0
        eng = self._engine()
        local = torch.cat(results, 0) if results else torch.empty((0, T), dtype=torch.float32, device=eng.device)
        return sharding.gather_assigned(local, mine, parts, group)

    # ------------------------------------------------------------------ loaders
    @classmethod
    def from_local(cls, ckpt_dir, device="cuda", precision: str = "fp16") -> "FlowHighSR":
        """flowhighsr.py:109-137: expects bigvgan_48khz_256band.{json,pt} and FLowHigh_basic_400k.pt."""
        ckpt_dir = Path(ckpt_dir)
        voc = MelVoco(vocoder_config=ckpt_dir / "bigvgan_48khz_256band.json",
                      vocoder_path=ckpt_dir / "bigvgan_48khz_256band.pt")
        net = FLowHigh(dim_in=voc.n_mels, audio_enc_dec=voc, depth=2)
        model = cls(flowhigh=net, precision=precision)  # defaults: basic_cfm / midpoint / sigma 0 (F4)
        ckpt = torch.load(ckpt_dir / "FLowHigh_basic_400k.pt", map_location="cpu")
        model.load_state_dict(ckpt["model"])
        return model.to(device).eval()

    @classmethod
    def from_pretrained(cls, device="cuda", precision: str = "fp16") -> "FlowHighSR":
        """flowhighsr.py:139-149 (needs network access to the HF hub)."""
        from huggingface_hub import hf_hub_download
        local_path = None
        for fpath in ["FLowHigh_basic_400k.json", "bigvgan_48khz_256band.json", "FLowHigh_basic_400k.pt",
                      "bigvgan_48khz_256band.pt"]:
            local_path = hf_hub_download(repo_id=REPO_ID, filename=fpath)
        return cls.from_local(Path(local_path).parent, device, precision=precision)

    @classmethod
    def from_random(cls, vcfg: Optional[VocoderConfig] = None, device="cuda", seed: int = 0, precision: str = "fp16",
                    vocoder_gain: float = 0.7, depth: int = 2, use_unet_skip_connection: bool = False,
                    architecture: str = "transformer", **kw) -> "FlowHighSR":
        """Random-init weights of the named architecture (no checkpoints offline)."""
        vcfg = vcfg or VocoderConfig.assumed_48k()
        voc = MelVoco(vocoder_config=vcfg)
        net = FLowHigh(dim_in=voc.n_mels, audio_enc_dec=voc, depth=depth, use_unet_skip_connection=use_unet_skip_connection,
                       architecture=architecture)
        model = cls(flowhigh=net, precision=precision, **kw)
        model.load_state_dict(random_state_dict(net.bcfg, vcfg, seed=seed, vocoder_gain=vocoder_gain))
        return model.to(device).eval()
