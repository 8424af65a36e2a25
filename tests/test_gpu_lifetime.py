"""Device memory is released by the objects that own it: repeated host-buffer front-end calls
reuse the context's scratch, and create -> use -> close cycles of every object type return free
device memory to where it started. Free memory is read device-wide, so the margins leave room for
other work on the same GPU."""

import numpy as np
import pytest

import pocketkaldi_b200 as pk
from pocketkaldi_b200 import formats
from pocketkaldi_b200.synth import synth_pcm

pytestmark = pytest.mark.gpu

MARGIN = 64 << 20


def free_bytes():
    import torch
    return torch.cuda.mem_get_info(0)[0]


@pytest.fixture(scope="module")
def ctx():
    c = pk.Context(0)
    yield c
    c.close()


def test_frontend_calls_do_not_leak(ctx, golden):
    pcm = synth_pcm(7, [0], 4000)[0]
    g = golden["cmvn_stats"]

    def calls(n):
        for _ in range(n):
            raw = ctx.fbank_batch([pcm])
            ctx.cmvn_batch(raw, g)

    calls(5)
    before = free_bytes()
    calls(200)
    assert before - free_bytes() <= MARGIN


def test_create_use_close_cycles_return_device_memory(ctx, golden, toy_conf):
    g = golden["cmvn_stats"]
    fst_path = formats.conf_path(toy_conf, formats.read_conf(toy_conf)["fst"])
    lens = [16000, 9000]
    pcm = np.concatenate([synth_pcm(11, [u], n)[0] for u, n in enumerate(lens)])
    S, chunk = 2, 2560
    chunks = synth_pcm(12, np.arange(S), chunk * 6)

    def cycle():
        am = pk.AcousticModel(ctx, pk.PREC_FP16R).Read(toy_conf)
        fst = pk.Fst(ctx, path=fst_path)
        b = pk.Batch(ctx, lens, g, am, prob_scale=0.1)
        b.set_pcm(pcm)
        b.run(pk.STAGE_ALL)
        b.set_compact(True)
        b.run(pk.STAGE_NNET)
        b.set_compact(False)
        b.run(pk.STAGE_NNET)
        hyps, _ = b.decode(fst)
        assert len(hyps) == len(lens)
        b.close()
        fst.close()
        st = pk.Stream(ctx, am, S, chunk, g, 0.1)
        buf = np.empty((S, chunk), np.int16)
        for k in range(6):  # the same host buffers from the third push on: the CUDA graph replays
            buf[:] = chunks[:, k * chunk:(k + 1) * chunk]
            st.push(buf)
        st.flush()
        st.close()
        ev = pk.Event(ctx)
        ev.record()
        ev.wait()
        ev.close()
        am.close()
        inner = pk.Context(0)
        inner.cmvn_batch(inner.fbank_batch([pcm[:16000]]), g)
        inner.flush_l2()  # 256 MiB of context scratch
        inner.close()

    cycle()
    before = free_bytes()
    for _ in range(20):
        cycle()
    assert before - free_bytes() <= MARGIN
