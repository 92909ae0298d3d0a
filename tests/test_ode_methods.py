"""GPU tests of torchdiffeq's `rk4` and `dopri5` (`torchdiffeq_ode_method`) through the public FlowHighSR surface: the
engine's solves against the oracle restatements (oracle/model.py, oracle/ode_torchdiffeq.py), per-clip equality of the
batched paths, CUDA-graph replay of the fixed-grid solve, and no capture of the adaptive one."""
import numpy as np
import pytest
import torch

from flowhigh_b200 import FlowHighSR
from flowhigh_b200.synth import synth_speech
from oracle import dsp, model, ode_torchdiffeq as otd
from util import golden_weights, load_golden, snr_db

pytestmark = pytest.mark.gpu


def _model(sd, vcfg, precision, **kw):
    m = FlowHighSR.from_random(vcfg, device="cuda:0", precision=precision, **kw)
    m.load_state_dict(sd)
    return m.cuda()


def _two_clips(n):
    g = load_golden("gen_basic_midpoint")
    sd, vcfg = golden_weights(g)
    cond = torch.from_numpy(np.ascontiguousarray(g["ref_cond_mel"]))[:, :n]
    cond = torch.cat([cond, cond.flip(1) * 0.8 - 1.0]).contiguous()
    eps = torch.from_numpy(np.ascontiguousarray(g["eps"])).reshape(1, -1, 256)[:, :n]
    eps = torch.cat([eps, eps.flip(2)]).contiguous()
    return sd, vcfg, cond, eps


def test_rk4_sample_f32_matches_oracle(cuda_device):
    sd, vcfg, cond, eps = _two_clips(48)
    m = _model(sd, vcfg, "fp32", torchdiffeq_ode_method="rk4")
    out = m.sample(cond=cond, time_steps=4, decode_to_audio=False, eps=eps).cpu()
    kw = dict(steps=4, ode_method="rk4", cfm_method="basic_cfm", sigma=0.0)
    ref64 = otd.cfm_sample_mel({k: v.double() for k, v in sd.items()}, cond.double(), eps.double(), **kw)
    ref32 = otd.cfm_sample_mel(sd, cond, eps, **kw)
    floor = float((ref32.double() - ref64).abs().max())
    e64 = float((out.double() - ref64).abs().max())
    print(f"rk4 fp32 sample: max-abs vs oracle fp64 {e64:.3g} (oracle fp32's own {floor:.3g})")
    assert e64 <= 3 * floor + 1e-4
    # and it is rk4, not the 4-step midpoint solve
    mid = otd.cfm_sample_mel(sd, cond, eps, **dict(kw, ode_method="midpoint"))
    assert float((mid.double() - ref64).abs().max()) > 10 * e64


def _mixed_rate_clips():
    """Three clips of 0.5 s at 12 / 16 / 24 kHz: one output length (24000 samples, 50 frames)."""
    return [(synth_speech(6000, 12000, seed=1), 12000), (synth_speech(8000, 16000, seed=2), 16000),
            (synth_speech(12000, 24000, seed=3), 24000)]


def test_rk4_generate_batch_per_clip_and_graph_replay(cuda_device):
    g = load_golden("gen_basic_midpoint")
    sd, vcfg = golden_weights(g)
    m = _model(sd, vcfg, "fp16", torchdiffeq_ode_method="rk4")
    clips = _mixed_rate_clips()
    gen = torch.Generator().manual_seed(4)
    eps = [torch.randn((1, 50, 256), generator=gen) for _ in clips]
    wavs, srs = [w for w, _ in clips], [s for _, s in clips]
    calls = [[o.cpu() for o in m.generate_batch(wavs, srs, eps=eps, timestep=2)] for _ in range(3)]
    assert len(m._graphs) == 1  # the third call replayed the captured graph
    for a, b in zip(calls[0], calls[2]):
        assert torch.equal(a, b)
    for (w, s), e, b in zip(clips, eps, calls[0]):
        one = m.generate(w, s, 48000, timestep=2, eps=e).cpu()
        assert torch.isfinite(one).all() and torch.equal(one, b)


def test_dopri5_sample_solves_the_batch_as_one_problem(cuda_device):
    sd, vcfg, cond, eps = _two_clips(32)
    tol = 1e-5
    m = _model(sd, vcfg, "fp32", torchdiffeq_ode_method="dopri5", ode_atol=tol, ode_rtol=tol)
    out = m.sample(cond=cond, time_steps=4, decode_to_audio=False, eps=eps).cpu()
    stats = m._engine().ode_stats
    sd64 = {k: v.double() for k, v in sd.items()}
    fn = lambda t, y: model.vector_field(sd64, y, cond.double(), t.double())
    ref64, st64 = otd.odeint_dopri5(fn, eps.double(), torch.linspace(0, 1, 5), atol=tol, rtol=tol)
    ref32 = otd.cfm_sample_mel(sd, cond, eps, steps=4, ode_method="dopri5", cfm_method="basic_cfm", sigma=0.0,
                                 atol=tol, rtol=tol)
    floor = float((ref32.double() - ref64[-1]).abs().max())
    e64 = float((out.double() - ref64[-1]).abs().max())
    print(f"dopri5 fp32 sample B=2: max-abs vs oracle fp64 {e64:.3g} (oracle fp32's own {floor:.3g}); GPU {stats}, "
          f"oracle {st64}")
    assert len(stats) == 1
    assert abs(stats[0]["n_steps"] - st64["n_steps"]) <= 1 and stats[0]["n_f_evals"] == 2 + 6 * stats[0]["n_steps"]
    assert e64 <= 3 * floor + 2e-3


def test_dopri5_generate_batch_is_per_clip_and_never_captured(cuda_device):
    g = load_golden("gen_basic_midpoint")
    sd, vcfg = golden_weights(g)
    m = _model(sd, vcfg, "fp16", torchdiffeq_ode_method="dopri5", ode_atol=1e-3, ode_rtol=1e-3)
    clips = _mixed_rate_clips()[:2]
    gen = torch.Generator().manual_seed(6)
    eps = [torch.randn((1, 50, 256), generator=gen) for _ in clips]
    for _ in range(3):
        outs = [o.cpu() for o in m.generate_batch([w for w, _ in clips], [s for _, s in clips], eps=eps)]
        stats = m._engine().ode_stats
    assert len(m._graphs) == 0 and len(stats) == 2
    for (w, s), e, b, st in zip(clips, eps, outs, stats):
        one = m.generate(w, s, 48000, eps=e).cpu()
        assert torch.isfinite(one).all() and torch.equal(one, b)
        assert m._engine().ode_stats == [st]


def _oracle_generate64(sd, vcfg, wav, sr, eps, **cfm):
    """oracle/pipeline.py's generate in fp64 with the torchdiffeq solvers of `ode_torchdiffeq.cfm_sample_mel`."""
    sd64 = {k: v.double() for k, v in sd.items()}
    cond = torch.from_numpy(np.ascontiguousarray(dsp.preprocess_audio(wav.astype(np.float64), sr, 48000))).float()[None]
    mel = otd.cfm_sample_mel(sd64, dsp.encode_logmel(cond), eps.double().reshape(1, -1, 256), steps=1,
                               cfm_method="basic_cfm", sigma=0.0, **cfm)
    return dsp.postprocess(model.vocoder_forward(sd64, vcfg, mel).squeeze(1), cond, cond.shape[-1]).float()


@pytest.mark.parametrize("method", ["rk4", "dopri5"])
def test_fp16_generate_matches_oracle_pipeline(cuda_device, method):
    g = load_golden("gen_basic_midpoint")
    sd, vcfg = golden_weights(g)
    m = _model(sd, vcfg, "fp16", torchdiffeq_ode_method=method, ode_atol=1e-3, ode_rtol=1e-3)
    wav, sr = g["wav"], int(g["sr"])
    eps = torch.from_numpy(g["eps"])
    out = m.generate(wav, sr, 48000, timestep=1, eps=eps).cpu()  # overflow_check = "raise": the guard is clean
    ref = _oracle_generate64(sd, vcfg, wav, sr, eps, ode_method=method, atol=1e-3, rtol=1e-3)
    print(f"{method} fp16 generate: SNR vs oracle fp64 {snr_db(ref, out):.1f} dB")
    assert out.shape == ref.shape and torch.isfinite(out).all() and snr_db(ref, out) >= 30.0


def test_unbuilt_torchdiffeq_methods_raise(cuda_device):
    g = load_golden("gen_basic_midpoint")
    sd, vcfg = golden_weights(g)
    m = _model(sd, vcfg, "fp32", torchdiffeq_ode_method="bosh3")
    with pytest.raises(ValueError, match="rk4"):
        m.generate(g["wav"], int(g["sr"]), 48000, eps=torch.from_numpy(g["eps"]))
