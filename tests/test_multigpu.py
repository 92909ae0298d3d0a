"""2-GPU NCCL tests of the sharded paths (run with `python -m pytest tests/test_multigpu.py -m gpu` on a machine with
at least two GPUs; skipped with one): distributed long-form chunks and sharded mixed-rate clips against the 1-GPU
calls, bit for bit."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu


def _model(dev):
    from flowhigh_b200 import FlowHighSR
    from util import golden_weights, load_golden
    g = load_golden("gen_basic_midpoint")
    sd, vcfg = golden_weights(g)
    m = FlowHighSR.from_random(vcfg, device=dev, precision="fp16")
    m.load_state_dict(sd)
    m = m.to(dev)
    m.cuda_graphs = False
    return m


def _worker(rank, world, port, q):
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dev = torch.device(f"cuda:{rank}")
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    from flowhigh_b200.synth import synth_speech
    m = _model(dev)
    res = {}
    # ---- long-form: 5.3 s at 16 kHz in 1 s chunks with 0.2 s overlap (7 chunks over 2 ranks: 4 + 3)
    wav = synth_speech(int(5.3 * 16000), 16000, seed=4)
    T = wav.shape[0] * 3
    clen, ov = 48000, 9600
    K = -(-(T - clen) // (clen - ov)) + 1
    eps = torch.randn((K, clen // 480, 256), generator=torch.Generator().manual_seed(3)).to(dev)
    kw = dict(timestep=1, chunk_seconds=1.0, overlap_seconds=0.2, eps=eps)
    multi = m.generate_long(wav, 16000, 48000, **kw)
    single = m.generate_long(wav, 16000, 48000, distributed=False, **kw)
    res["long_equal"] = bool(torch.equal(multi, single)) and bool(torch.isfinite(multi).all())
    res["long_shape"] = tuple(multi.shape)
    # ---- sharded mixed-rate clips, gathered with one all_gather_into_tensor
    rates = [8000, 12000, 16000, 24000]
    srs = [rates[i % 4] for i in range(7)]
    audios = [synth_speech(sr // 2, sr, seed=10 + i) for i, sr in enumerate(srs)]  # 0.5 s each -> 24000 samples out
    e = [torch.randn((50, 256), generator=torch.Generator().manual_seed(20 + i)).to(dev) for i in range(7)]
    got = m.generate_sharded(audios, srs, 48000, timestep=1, eps=e, gather=True)
    want = torch.cat(m.generate_batch(audios, srs, 48000, timestep=1, eps=e), 0)
    res["shard_equal"] = bool(torch.equal(got, want))
    res["shard_shape"] = tuple(got.shape)
    t = torch.tensor([float(rank + 1)], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    res["max"] = float(t)
    q.put((rank, res))
    dist.destroy_process_group()


def test_two_rank_nccl_long_form_and_sharded_clips():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    out = [q.get(timeout=600) for _ in procs]
    for p in procs:
        p.join(timeout=120)
    for rank, res in out:
        print(rank, res)
        assert res["long_equal"] and res["shard_equal"] and res["max"] == 2.0, (rank, res)
        assert res["shard_shape"] == (7, 24000)
