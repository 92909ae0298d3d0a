"""Clips of different input rates with one output length share a batch (generate_batch / generate_sharded group by
output length): one pass of every kernel behind the resampler, and every clip bit-identical to its own `generate` on
the 16-bit paths.  Run with -m gpu on a B200."""
import numpy as np
import pytest
import torch

from flowhigh_b200 import FlowHighSR
from flowhigh_b200.engine import Engine
from flowhigh_b200.synth import synth_speech
from util import golden_weights, load_golden

pytestmark = pytest.mark.gpu

RATES = [8000, 12000, 16000, 24000]


@pytest.fixture(scope="module")
def model():
    """model(precision) -> FlowHighSR with the golden fixture's weights, one per precision for the module."""
    g = load_golden("gen_basic_midpoint")
    sd, vcfg = golden_weights(g)
    cache = {}

    def get(precision):
        if precision not in cache:
            m = FlowHighSR.from_random(vcfg, device="cuda:0", precision=precision)
            m.load_state_dict(sd)
            cache[precision] = m.cuda()
        m = cache[precision]
        m.cuda_graphs, m.upsampling_method = False, "scipy"
        return m
    return get


def _clips(n, seconds=0.25, seed=0):
    """n clips cycling through 8 / 12 / 16 / 24 kHz, all `seconds` long (one output length), different gains."""
    srs = [RATES[i % 4] for i in range(n)]
    wavs = [synth_speech(int(seconds * sr), sr, seed=seed + i) * (0.3 + 0.05 * i) for i, sr in enumerate(srs)]
    return wavs, srs


def _eps(T_out, seed):
    return torch.from_numpy(np.random.default_rng(seed).standard_normal((T_out // 480, 256)).astype(np.float32))


def _per_clip(m, wavs, srs, eps):
    return [m.generate(w, s, 48000, timestep=1, eps=e) for w, s, e in zip(wavs, srs, eps)]


def test_resample_normalise_parts_equals_per_part(cuda_device, model):
    """Row offsets, the 48 kHz copy and the shared normalisation of a multi-part batch against each part alone.  The filter
    itself is checked against scipy / the soxr_hq design by test_resample_normalise and test_soxr_hq_resample_normalise."""
    eng = model("fp32")._engine()
    parts = [(synth_speech(n, sr, seed=sr)[None].repeat(2, 0) * np.float32([[0.5], [2.0]]), sr)
             for sr, n in ((8000, 4000), (48000, 24000), (22050, 11025), (16000, 8000))]
    dev = [(torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).cuda(), sr) for x, sr in parts]
    for method in ("scipy", "soxr_hq"):
        got = eng.resample_normalise_parts(dev, 48000, method=method)
        want = torch.cat([eng.resample_normalise(x, sr, method=method) for x, sr in dev])
        assert got.shape == (8, 24000) and torch.equal(got, want), method
    with pytest.raises(ValueError):
        eng.resample_normalise_parts([dev[0], (dev[1][0][:, :-1].contiguous(), 48000)], 48000)


def test_mixed_rates_run_as_one_batch(cuda_device, model, monkeypatch):
    m = model("fp16")
    seen = {"encode": [], "vocoder": []}
    for name in seen:
        orig = getattr(Engine, name)

        def rec(self, x, *a, _orig=orig, _name=name, **k):
            seen[_name].append(int(x.shape[0]))
            return _orig(self, x, *a, **k)
        monkeypatch.setattr(Engine, name, rec)
    wavs, srs = _clips(8)
    outs = m.generate_batch(wavs, srs, 48000, timestep=1)
    assert seen == {"encode": [8], "vocoder": [8]}
    assert all(o.shape == (1, 12000) and torch.isfinite(o).all() for o in outs)


@pytest.mark.parametrize("precision", ["fp16", "fp16x2", "fp32"])
@pytest.mark.parametrize("n", [3, 9])  # both sides of the B <= 4 parallel-AMP-branch threshold
def test_mixed_rate_batch_equals_per_clip(cuda_device, model, precision, n):
    m = model(precision)
    wavs, srs = _clips(n, seed=10 * n)
    eps = [_eps(12000, seed=100 * n + i) for i in range(n)]
    outs = m.generate_batch(wavs, srs, 48000, timestep=1, eps=eps)
    for i, single in enumerate(_per_clip(m, wavs, srs, eps)):
        assert outs[i].shape == single.shape == (1, 12000)
        if precision == "fp32":
            assert float((outs[i] - single).abs().max()) <= 2e-5, i
        else:
            assert torch.equal(outs[i], single), (i, float((outs[i] - single).abs().max()))


def test_mixed_input_lengths_in_one_group(cuda_device, model):
    """One output length (24000 samples) from five input lengths and rates, among them a 48 kHz clip (no resampling, copied
    into the batch) and a clip in int16 range (max > 1: the /32768 path)."""
    m = model("fp16")
    spec = [(8000, 4000), (16000, 8000), (48000, 24000), (22050, 11025), (16000, 8000), (12000, 6000), (8000, 4000)]
    wavs = [synth_speech(n, sr, seed=i) * (0.4 + 0.05 * i) for i, (sr, n) in enumerate(spec)]
    wavs[4] = wavs[4] * 20000.0
    srs = [sr for sr, _ in spec]
    eps = [_eps(24000, seed=i) for i in range(len(spec))]
    outs = m.generate_batch(wavs, srs, 48000, timestep=1, eps=eps)
    for i, single in enumerate(_per_clip(m, wavs, srs, eps)):
        assert outs[i].shape == (1, 24000) and torch.equal(outs[i], single), i


def test_mixed_rates_librosa_branch(cuda_device, model):
    m = model("fp16")
    m.upsampling_method = "librosa"
    wavs, srs = _clips(6, seed=40)
    eps = [_eps(12000, seed=40 + i) for i in range(6)]
    outs = m.generate_batch(wavs, srs, 48000, timestep=1, eps=eps)
    for i, single in enumerate(_per_clip(m, wavs, srs, eps)):
        assert torch.equal(outs[i], single), i
    m.upsampling_method = "scipy"
    scipy_out = m.generate_batch(wavs, srs, 48000, timestep=1, eps=eps)
    assert not torch.equal(scipy_out[1], outs[1])  # the librosa taps were really used


def test_every_host_path_matches_pageable_eager(cuda_device, model):
    """CUDA-graph capture + replay, page-locked staging, direct page-locked tensors, out_host with chunked read-back and
    with two sub-batches: all bit-identical to the pageable eager call, results in caller order."""
    m = model("fp16")
    wavs, srs = _clips(8, seed=60)
    wavs[5] = wavs[5] * 20000.0  # int16 range: skipped by the direct path, cancelled by the peak normalisation
    eps = [_eps(12000, seed=60 + i) for i in range(8)]
    ref = m.generate_batch(wavs, srs, 48000, timestep=1, eps=eps)

    m.cuda_graphs = True
    n_graphs = len(m._graphs)
    for _ in range(3):  # first sighting eager, second captures + replays, third replays
        got = m.generate_batch(wavs, srs, 48000, timestep=1, eps=eps)
        assert all(torch.equal(a, b) for a, b in zip(ref, got))
    assert len(m._graphs) == n_graphs + 1
    assert next(reversed(m._graphs))[0] == ((8000, 2000, 2), (12000, 3000, 2), (16000, 4000, 2), (24000, 6000, 2))
    m.cuda_graphs = False

    got = m.generate_batch(wavs, srs, 48000, timestep=1, eps=eps, pinned=True)
    assert all(torch.equal(a, b) for a, b in zip(ref, got))

    host = [torch.from_numpy(np.asarray(w, dtype=np.float32)).pin_memory() for w in wavs]
    got = m.generate_batch(host, srs, 48000, timestep=1, eps=eps, pinned=True)
    assert all(torch.equal(a, b) for a, b in zip(ref, got))

    old = m.readback_chunk, m.overlap_min_batch
    try:
        for chunk, overlap in ((2, 1 << 30), (16, 3)):
            m.readback_chunk, m.overlap_min_batch = chunk, overlap
            out_host = torch.zeros((8, 12000), dtype=torch.float32).pin_memory()
            got = m.generate_batch(host, srs, 48000, timestep=1, eps=eps, pinned=True, out_host=out_host)
            torch.cuda.synchronize()
            for i in range(8):
                assert torch.equal(ref[i], got[i]) and torch.equal(out_host[i: i + 1], ref[i].cpu()), (chunk, overlap, i)
    finally:
        m.readback_chunk, m.overlap_min_batch = old


def test_different_output_lengths_keep_caller_order(cuda_device, model):
    m = model("fp16")
    spec = [(8000, 2000), (16000, 8000), (12000, 3000), (24000, 12000), (48000, 12000), (16000, 4000), (8000, 4000)]
    wavs = [synth_speech(n, sr, seed=70 + i) * 0.5 for i, (sr, n) in enumerate(spec)]
    srs = [sr for sr, _ in spec]
    T = [n * 48000 // sr for sr, n in spec]
    eps = [_eps(t, seed=70 + i) for i, t in enumerate(T)]
    outs = m.generate_batch(wavs, srs, 48000, timestep=1, eps=eps)
    for i, single in enumerate(_per_clip(m, wavs, srs, eps)):
        assert outs[i].shape == (1, T[i]) and torch.equal(outs[i], single), i


def test_generate_sharded_one_rank_batches_mixed_rates(cuda_device, model, monkeypatch):
    """generate_sharded on one process: one generate_batch call per output length and max_batch slice, results in clip
    order and equal to generate_batch."""
    m = model("fp16")
    wavs, srs = _clips(10, seed=80)
    eps = [_eps(12000, seed=80 + i) for i in range(10)]
    want = torch.cat(m.generate_batch(wavs, srs, 48000, timestep=1, eps=eps))
    calls = []
    orig = FlowHighSR.generate_batch

    def rec(self, audios, sr, *a, **k):
        calls.append(list(sr))
        return orig(self, audios, sr, *a, **k)
    monkeypatch.setattr(FlowHighSR, "generate_batch", rec)
    got = m.generate_sharded(wavs, srs, 48000, timestep=1, eps=eps, max_batch=6)
    assert torch.equal(got, want)
    assert [len(c) for c in calls] == [6, 4] and sorted(sum(calls, [])) == sorted(srs)
