"""Lattices of the online GPU decoder (pkb_decoder_set_lattice / _lattice / _lattice_get): whatever the
split of the rows into advances or pushes, each finish must leave, per stream, the records and best
cost of pkb_batch_lattice over the same rows, bit for bit, and switching lattices on must change
nothing else the decoder returns. A lattice that does not fit fails only its own stream's lattice."""

import math
import os
import sys

import numpy as np
import pytest

import pocketkaldi_b200 as pk
import tools.decode_demo as demo
from oracle.decoder import host_viterbi
from pocketkaldi_b200 import formats
from pocketkaldi_b200.synth import synth_global_cmvn

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from test_gpu_lattice import LENS, batch_of, host_lattice, same_records  # noqa: E402
from test_gpu_online_decode import (MARGIN, decode_in_splits, host_record_counts, make_model,  # noqa: E402
                                    one_word_rows, run_child)
from test_gpu_viterbi import coloured  # noqa: E402

BEAMS = (0.5, 4.0, math.inf)


@pytest.fixture(scope="module")
def ctx():
    c = pk.Context(0)
    yield c
    c.close()


def raw_lattice(dec):
    """pkb_decoder_lattice's codes and best costs, without the records."""
    na = np.zeros(dec.n_streams, np.int64)
    best = np.zeros(dec.n_streams, np.float64)
    pk.binding._check(dec.ctx.lib.pkb_decoder_lattice(dec.h, na.ctypes.data, best.ctypes.data))
    return na, best


def assert_same_lattices(got, want, what):
    (gl, gb), (wl, wb) = got, want
    assert len(gl) == len(wl)
    for s, (g, w) in enumerate(zip(gl, wl)):
        assert (g is None) == (w is None), (what, s)
        assert g is None or same_records(g, w), (what, s, None if g is None else len(g), None if w is None else len(w))
    assert gb.tobytes() == wb.tobytes(), (what, gb, wb)


# ---------------------------------------------------------------- split invariance
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["loop", "eps", "loop_mid", "loop_big"])
def test_split_invariance_bitwise_against_batch_lattice(ctx, kind):
    am, fst, _, _ = make_model(ctx, kind)
    lens = LENS + [0]
    utts = []   # two utterances in a row through the same decoder: nothing may carry over
    for seed in (100, 900):
        b, rows = batch_of(ctx, am, lens, seed=seed)
        hyps, wts = b.decode(fst)
        lats = {lb: b.lattice(fst, lattice_beam=lb) for lb in BEAMS}
        b.close()
        assert any(len(x) > 0 for x in lats[4.0][0])
        utts.append((rows, hyps, wts, lats))
    T = max(r.shape[0] for u in utts for r in u[0])
    for lb in BEAMS:
        for k in (1, 7, 16, T):
            dec = pk.Decoder(ctx, am, fst, len(lens))
            dec.set_lattice(lb, max_frames=T)   # the default max_arcs is then the batch's
            for rows, hyps, wts, lats in utts:
                got, gw = decode_in_splits(dec, rows, k)
                assert got == hyps, (kind, lb, k)
                assert gw.tobytes() == wts.tobytes(), (kind, lb, k)
                assert_same_lattices(dec.lattice(), lats[lb], (kind, lb, k))
            dec.close()
    fst.close()
    am.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["loop", "eps", "loop_big"])
def test_lattices_change_nothing_else(ctx, kind):
    am, fst, _, _ = make_model(ctx, kind)
    _, rows = batch_of(ctx, am, LENS, seed=200)
    for k in (1, 7):
        decs = [pk.Decoder(ctx, am, fst, len(LENS)) for _ in range(2)]
        decs[1].set_lattice(4.0, max_frames=max(r.shape[0] for r in rows))
        parts = [[], []]
        for i, d in enumerate(decs):
            parts[i].append(d.partial())
            res = decode_in_splits(d, rows, k, lambda t, i=i, d=d: parts[i].append(d.partial()))
            parts[i].append(res)
        assert len(parts[0]) == len(parts[1]) > 2
        for a, b in zip(parts[0], parts[1]):
            assert a[0] == b[0]
            for x, y in zip(a[1:], b[1:]):
                assert x.tobytes() == y.tobytes()
        for d in decs:
            d.close()
    fst.close()
    am.close()


# ---------------------------------------------------------------- attached to a stream
def stream_rows(st, pcm, chunk, rows):
    """Pushes pcm [S][n] chunk by chunk and flushes; returns each stream's rows (rows=True) or None."""
    out = []
    for k in range(pcm.shape[1] // chunk):
        o = st.push(pcm[:, k * chunk:(k + 1) * chunk], rows=rows)
        if rows:
            out.append(o.copy())
    o = st.flush(rows=rows)
    if not rows:
        return None
    out.append(o.copy())
    cat = np.concatenate(out, axis=1)
    return [cat[s] for s in range(pcm.shape[0])]


def check_attached_stream(chunk):
    ctx = pk.Context(0)
    am, fst, graph, tid2pdf = make_model(ctx, "loop")
    S, n = 5, 64000
    st = pk.Stream(ctx, am, S, chunk, synth_global_cmvn(), 0.1)
    dec = pk.Decoder(ctx, am, fst, S)
    ref = pk.Decoder(ctx, am, fst, S)
    ref.set_lattice(4.0)
    st.set_decoder(dec)
    graphs = os.environ.get("PKB_STREAM_GRAPH") != "0"
    # an utterance without lattices: from the fourth push on the pushes replay captured graphs
    steady = graphs and n // chunk >= 4
    pcm0 = np.stack([coloured(800 + s, n) for s in range(S)])
    r0 = st.graph_replays()
    stream_rows(st, pcm0, chunk, rows=False)
    plain = dec.finish()
    assert (st.graph_replays() > r0) == steady
    with pytest.raises(pk.PkbError):
        dec.lattice()     # that finish ran without lattices
    # switched on after the capture, with the same host buffers: the decode-only pushes right after
    # must not replay a graph without the lattice work
    dec.set_lattice(4.0)
    for rep in range(2):
        pcm = np.stack([coloured(810 + 10 * rep + s, n) for s in range(S)])
        r0 = st.graph_replays()
        stream_rows(st, pcm, chunk, rows=False)   # decode-only pushes
        only = dec.finish()
        lat_only = dec.lattice()
        assert (st.graph_replays() > r0) == steady
        rows = stream_rows(st, pcm, chunk, rows=True)
        with_rows = dec.finish()
        lat_rows = dec.lattice()
        assert only[0] == with_rows[0] and only[1].tobytes() == with_rows[1].tobytes()
        assert_same_lattices(lat_only, lat_rows, ("decode-only", chunk, rep))
        ref.advance(np.stack(rows))
        want = ref.finish()
        assert want[0] == only[0] and want[1].tobytes() == only[1].tobytes()
        assert_same_lattices(lat_only, ref.lattice(), ("host-fed", chunk, rep))
        for s in range(S):
            h, hbest, _ = host_lattice(graph, tid2pdf, rows[s], lattice_beam=4.0)
            assert same_records(lat_only[0][s], h), (chunk, rep, s)
            assert np.float64(lat_only[1][s]).tobytes() == np.float64(hbest).tobytes()
        assert all(len(x) > 0 for x in lat_only[0])
    assert plain[0] is not None
    for o in (st, dec, ref, fst, am):
        o.close()
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [160, 2560, 16000])
def test_attached_stream_lattices(chunk):
    check_attached_stream(chunk)


@pytest.mark.gpu
def test_attached_stream_lattices_eager():
    run_child("import test_gpu_online_lattice as t\nfor c in (160, 2560, 16000):\n    t.check_attached_stream(c)\n"
              "print('CHILD OK')", PKB_STREAM_GRAPH="0")


# ---------------------------------------------------------------- limits and errors
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["loop", "loop_big"])
def test_frame_and_arc_limits_fail_only_the_long_stream(ctx, kind):
    am, fst, graph, tid2pdf = make_model(ctx, kind)
    b, rows = batch_of(ctx, am, LENS)
    hyps, wts = b.decode(fst)
    full = b.lattice(fst, lattice_beam=4.0)
    T = [r.shape[0] for r in rows]
    n_log = [host_lattice(graph, tid2pdf, r, lattice_beam=4.0)[2] for r in rows]
    big, longest = int(np.argmax(n_log)), int(np.argmax(T))
    assert sorted(n_log)[-2] < n_log[big] and sorted(T)[-2] < T[longest]
    capped = b.lattice(fst, lattice_beam=4.0, max_arcs=n_log[big] - 1)
    b.close()
    assert capped[0][big] is None
    for max_frames, max_arcs, bad, code, want in ((T[longest] - 1, 0, longest, -5, full),
                                                   (T[longest], n_log[big] - 1, big, -4, capped)):
        dec = pk.Decoder(ctx, am, fst, len(LENS))
        dec.set_lattice(4.0, max_frames=max_frames, max_arcs=max_arcs)
        for k in (7, 16):
            got, gw = decode_in_splits(dec, rows, k)
            assert got == hyps and gw.tobytes() == wts.tobytes(), (kind, code, k)
            na, best = raw_lattice(dec)
            assert na[bad] == code and best[bad] == math.inf, (kind, code, k, na)
            lats = dec.lattice()
            for s in range(len(LENS)):
                if s == bad:
                    assert lats[0][s] is None
                else:
                    assert same_records(lats[0][s], want[0][s]), (kind, code, k, s)
                    assert np.float64(lats[1][s]).tobytes() == np.float64(want[1][s]).tobytes()
        dec.close()
    fst.close()
    am.close()


@pytest.mark.gpu
def test_token_overflow_is_reported_and_the_next_utterance_is_clean(ctx):
    rng = np.random.default_rng(3)
    P = 640
    layers = formats.make_dnn(rng, 440, 32, 1, P)
    prior = np.full(P, 1.0 / P, np.float32)
    graph, tid2pdf = demo.word_loop_graph(200, 3, P)   # 601 states: table kernel, global tables
    am = pk.AcousticModel(ctx, pk.PREC_BF16X3).from_layers(layers, prior, 5, 5, tid2pdf=tid2pdf)
    fst = pk.Fst(ctx, graph=graph)
    from pocketkaldi_b200.synth import synth_pcm
    pcms = [synth_pcm(5, [0], 16000)[0], synth_pcm(5, [1], 16000)[0]]
    b = pk.Batch(ctx, [16000, 16000], synth_global_cmvn(), am, prob_scale=0.1)
    b.set_pcm(np.ascontiguousarray(np.concatenate(pcms), np.int16))
    b.run(pk.STAGE_ALL)
    ll = b.get(pk.BUF_LOGLIK)
    rows = [ll[:b.num_frames[0]], ll[b.num_frames[0]:]]
    b.close()
    dec = pk.Decoder(ctx, am, fst, 2, max_tokens=64)
    dec.set_lattice(4.0)
    hyps, _ = decode_in_splits(dec, rows, 16)
    assert hyps == [None, None]
    na, best = raw_lattice(dec)
    assert list(na) == [-1, -1] and np.all(best == math.inf)
    assert dec.lattice()[0] == [None, None]
    clean = one_word_rows(P, 600, 7, 30)
    hyps, _ = decode_in_splits(dec, [clean, clean], 16)
    assert hyps == [[8], [8]]
    want, wbest, _ = host_lattice(graph, tid2pdf, clean, lattice_beam=4.0)
    lats, best = dec.lattice()
    for s in range(2):
        assert same_records(lats[s], want) and best[s] == wbest
    dec.close()
    fst.close()
    am.close()


@pytest.mark.gpu
def test_a_failed_search_past_max_frames_leaves_the_other_streams_exact(ctx):
    # streams 1 and 3 (one of them the last) overflow their tokens early and then run past
    # max_frames: their lattices fail with the search's code, and neither may touch the lattice
    # state of a neighbour at the finish
    rng = np.random.default_rng(3)
    P = 640
    layers = formats.make_dnn(rng, 440, 32, 1, P)
    prior = np.full(P, 1.0 / P, np.float32)
    graph, tid2pdf = demo.word_loop_graph(200, 3, P)   # 601 states: table kernel, global tables
    am = pk.AcousticModel(ctx, pk.PREC_BF16X3).from_layers(layers, prior, 5, 5, tid2pdf=tid2pdf)
    fst = pk.Fst(ctx, graph=graph)
    from pocketkaldi_b200.synth import synth_pcm
    pcms = [synth_pcm(5, [0], 16000)[0], synth_pcm(5, [1], 16000)[0]]
    b = pk.Batch(ctx, [16000, 16000], synth_global_cmvn(), am, prob_scale=0.1)
    b.set_pcm(np.ascontiguousarray(np.concatenate(pcms), np.int16))
    b.run(pk.STAGE_ALL)
    ll = b.get(pk.BUF_LOGLIK)
    noisy = [ll[:b.num_frames[0]], ll[b.num_frames[0]:]]
    b.close()
    clean = [one_word_rows(P, 600, w, 30) for w in (7, 11)]
    max_frames = 40
    assert min(r.shape[0] for r in noisy) > max_frames + 16
    wants = [host_lattice(graph, tid2pdf, r, lattice_beam=4.0) for r in clean]
    words = [host_viterbi(graph, tid2pdf, r)[0] for r in clean]
    dec = pk.Decoder(ctx, am, fst, 4, max_tokens=64)
    dec.set_lattice(4.0, max_frames=max_frames)
    for rep in range(2):
        for k in (1, 16):
            hyps, _ = decode_in_splits(dec, [clean[0], noisy[0], clean[1], noisy[1]], k)
            assert hyps == [words[0], None, words[1], None] and all(words), (hyps, words)
            na, best = raw_lattice(dec)
            assert na[1] == -1 and na[3] == -1, na   # the token overflow came first
            lats, best = dec.lattice()
            for s, (want, wbest, _) in zip((0, 2), wants):
                assert same_records(lats[s], want), (rep, k, s)
                assert np.float64(best[s]).tobytes() == np.float64(wbest).tobytes()
    dec.close()
    fst.close()
    am.close()


@pytest.mark.gpu
def test_invalid_uses_are_rejected(ctx):
    am, fst, _, _ = make_model(ctx, "loop")
    S = 2
    dec = pk.Decoder(ctx, am, fst, S)
    rows = np.zeros((S, 4, am.num_pdfs()), np.float32)
    for lb in (-1.0, float("nan"), -math.inf):
        with pytest.raises(pk.PkbError):
            dec.set_lattice(lb)
    with pytest.raises(pk.PkbError):
        dec.set_lattice(4.0, max_arcs=2 ** 31 - 1)   # the log count must not wrap
    with pytest.raises(pk.PkbError):
        dec.lattice()                 # no finish yet
    dec.set_lattice(4.0)
    dec.advance(rows)
    with pytest.raises(pk.PkbError):
        dec.set_lattice(2.0)          # mid-utterance
    with pytest.raises(pk.PkbError):
        dec.set_lattice(0.0)
    dec.finish()
    lats, best = dec.lattice()
    assert all(x is not None for x in lats)
    dec.advance(rows)
    with pytest.raises(pk.PkbError):
        dec.lattice()                 # the next advance invalidates the results
    dec.finish()
    dec.set_lattice(0.0)              # off between utterances: the next finish has no lattice
    dec.advance(rows)
    dec.finish()
    with pytest.raises(pk.PkbError):
        dec.lattice()
    # attached: a push or flush invalidates the results too
    chunk = 2560
    st = pk.Stream(ctx, am, S, chunk, synth_global_cmvn(), 0.1)
    st.set_decoder(dec)
    dec.set_lattice(4.0)
    pcm = np.stack([coloured(950 + s, chunk) for s in range(S)])
    st.push(pcm, rows=False)
    with pytest.raises(pk.PkbError):
        dec.set_lattice(2.0)
    st.flush(rows=False)
    dec.finish()
    dec.lattice()
    st.push(pcm, rows=False)
    with pytest.raises(pk.PkbError):
        dec.lattice()
    st.flush(rows=False)
    dec.finish()
    for o in (st, dec, fst, am):
        o.close()


@pytest.mark.gpu
def test_long_stream_with_record_compaction(ctx):
    am, fst, graph, tid2pdf = make_model(ctx, "loop")
    _, rows = batch_of(ctx, am, [120 * 16000], seed=500)
    every = 16
    appended, live_max, adv_max = host_record_counts(graph, tid2pdf, rows[0], every)
    max_records = max(2 * live_max, 2 * adv_max)
    assert max_records <= appended // 4, (max_records, appended)   # the store is compacted
    T = rows[0].shape[0]
    dec = pk.Decoder(ctx, am, fst, 1, max_records=max_records)
    dec.set_lattice(4.0, max_frames=T)
    hyps, _ = decode_in_splits(dec, rows, every)
    assert hyps[0] is not None and len(hyps[0]) > 16
    want, wbest, _ = host_lattice(graph, tid2pdf, rows[0], lattice_beam=4.0)
    lats, best = dec.lattice()
    assert same_records(lats[0], want) and np.float64(best[0]).tobytes() == np.float64(wbest).tobytes()
    dec.close()
    fst.close()
    am.close()


@pytest.mark.gpu
def test_lattice_cycles_do_not_leak(ctx):
    import torch
    am, fst, _, _ = make_model(ctx, "loop")
    S, chunk = 4, 2560
    g = synth_global_cmvn()
    pcm = np.stack([coloured(970 + s, chunk) for s in range(S)])

    def cycle():
        st = pk.Stream(ctx, am, S, chunk, g, 0.1)
        dec = pk.Decoder(ctx, am, fst, S)
        dec.set_lattice(4.0, max_frames=200)
        st.set_decoder(dec)
        for _ in range(5):
            st.push(pcm, rows=False)
        st.flush(rows=False)
        dec.finish()
        lats, _ = dec.lattice()
        assert all(x is not None and len(x) for x in lats)
        dec.close()
        st.close()

    cycle()
    before = torch.cuda.mem_get_info(0)[0]
    for _ in range(20):
        cycle()
    assert before - torch.cuda.mem_get_info(0)[0] <= MARGIN
    fst.close()
    am.close()
