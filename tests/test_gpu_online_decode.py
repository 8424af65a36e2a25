"""Online GPU decoding (pkb_decoder_*): the resumable Viterbi search must give, for any split of the
rows into advances, bit-identical words and weight to one pkb_batch_decode over the same rows; its
best-so-far results must follow a host restatement of the search frame by frame; attached to a
stream it must decode during the push (also without copying rows back, inside the captured CUDA
graph); its word-record store must be compacted to what the live tokens reach."""

import os
import subprocess
import sys

import numpy as np
import pytest

import pocketkaldi_b200 as pk
import tools.decode_demo as demo
from oracle.decoder import host_viterbi
from pocketkaldi_b200 import formats
from pocketkaldi_b200.synth import synth_global_cmvn

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
from test_gpu_viterbi import coloured, eps_graph  # noqa: E402

MARGIN = 64 << 20
LENS = [16000, 24000, 8000, 32000, 400, 12345]


@pytest.fixture(scope="module")
def ctx():
    c = pk.Context(0)
    yield c
    c.close()


def make_model(ctx, kind):
    """(am, fst, graph, tid2pdf) for the graph kinds of test_gpu_viterbi.py, with acoustic scores
    made decisive the same way: "loop" 12 words (dense kernel), "eps" the epsilon hub, "loop_big"
    180 words / 541 states (table kernel, global tables), "loop_mid" 100 words / 301 states (table
    kernel, shared-memory tables)."""
    rng = np.random.default_rng({"loop": 1, "eps": 2, "loop_big": 3, "loop_mid": 4}[kind])
    P = 600 if kind in ("loop_big", "loop_mid") else 96
    layers = formats.make_dnn(rng, 440, 96, 2, P)
    layers[-2] = ("linear", (layers[-2][1] * 3.0).astype(np.float32), layers[-2][2])
    prior = rng.uniform(0.5, 1.5, P).astype(np.float32)
    prior /= prior.sum()
    if kind == "eps":
        graph, tid2pdf = eps_graph(10, 3, P)
    else:
        graph, tid2pdf = demo.word_loop_graph({"loop": 12, "loop_big": 180, "loop_mid": 100}[kind], 3, P)
    am = pk.AcousticModel(ctx, pk.PREC_BF16X3).from_layers(layers, prior, 5, 5, tid2pdf=tid2pdf)
    fst = pk.Fst(ctx, graph=graph)
    return am, fst, graph, tid2pdf


def batch_rows(ctx, am, fst, pcms):
    """pkb_batch_decode of the utterances and the batch's own log-likelihood rows per utterance."""
    b = pk.Batch(ctx, [len(p) for p in pcms], synth_global_cmvn(), am, prob_scale=0.1)
    b.set_pcm(np.ascontiguousarray(np.concatenate(pcms), np.int16))
    b.run(pk.STAGE_ALL)
    hyps, wts = b.decode(fst)
    ll = b.get(pk.BUF_LOGLIK)
    off = np.concatenate([[0], np.cumsum(b.num_frames)])
    rows = [ll[off[u]:off[u + 1]].copy() for u in range(len(pcms))]
    b.close()
    return hyps, wts, rows


def padded(rows):
    T = max(r.shape[0] for r in rows)
    out = np.zeros((len(rows), max(T, 1), rows[0].shape[1]), np.float32)
    for s, r in enumerate(rows):
        out[s, :r.shape[0]] = r
    return out


def decode_in_splits(dec, rows, k, each=None):
    """Feeds rows[s] to stream s, k frames per advance; `each(t)` runs after every advance."""
    T = np.array([r.shape[0] for r in rows])
    pad = padded(rows)
    for t0 in range(0, int(T.max()), k):
        dec.advance(pad[:, t0:t0 + k], np.clip(T - t0, 0, k))
        if each is not None:
            each(t0 + k)
    return dec.finish()


def test_loop_mid_takes_the_table_kernel_with_shared_memory_tables():
    # plan_viterbi (decoder.cu): more than 4096 arcs rule out the dense kernel, at most 512 states
    # put the token tables in shared memory (the graph of make_model(ctx, "loop_mid"))
    num_states, _, _, arcs = demo.word_loop_graph(100, 3, 600)[0]
    assert num_states <= 512 and len(arcs) > 4096


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["loop", "eps", "loop_big", "loop_mid"])
def test_split_invariance_bitwise_against_batch_decode(ctx, kind):
    am, fst, _, _ = make_model(ctx, kind)
    pcms = [coloured(100 + u, n) for u, n in enumerate(LENS)]
    hyps, wts, rows = batch_rows(ctx, am, fst, pcms)
    assert all(h is not None for h in hyps) and any(len(h) > 2 for h in hyps)
    for k in (1, 7, 16, max(r.shape[0] for r in rows)):
        dec = pk.Decoder(ctx, am, fst, len(pcms))
        got, gw = decode_in_splits(dec, rows, k)
        assert got == hyps, (kind, k)
        assert np.array_equal(gw.view(np.int32), wts.view(np.int32)), (kind, k, gw, wts)
        dec.close()


def run_child(code, **env):
    e = dict(os.environ)
    e.update(env)
    r = subprocess.run([sys.executable, "-c", "import sys; sys.path[:0] = [%r, %r]\n" % (ROOT, HERE) + code],
                       cwd=ROOT, env=e, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=900)
    assert r.returncode == 0, r.stdout.decode()[-4000:]
    assert b"CHILD OK" in r.stdout


# ---------------------------------------------------------------- host restatement with its tokens
def host_frames(graph, tid2pdf, loglik, beam=16.0):
    """oracle/decoder.host_viterbi's arithmetic, yielding the tokens {state: (cost, words)} after
    every frame."""
    num_states, start, finals, arcs = graph
    out = [[] for _ in range(num_states)]
    for src, dst, il, ol, w in arcs:
        out[src].append((dst, il, ol, float(np.float32(w))))
    f32 = lambda x: float(np.float32(x))

    def close(toks, cutoff):
        queue = list(toks)
        while queue:
            s = queue.pop()
            cost, words = toks[s]
            for dst, il, ol, w in out[s]:
                if il != 0 or cost + w > cutoff:
                    continue
                c = f32(cost + w)
                if dst not in toks or c < toks[dst][0]:
                    toks[dst] = (c, words + (ol,) if ol else words)
                    queue.append(dst)

    toks = {start: (0.0, ())}
    close(toks, np.inf)
    for row in loglik:
        if not toks:
            yield toks
            continue
        weight_cutoff = f32(min(c for c, _ in toks.values()) + beam)
        cand = [(cost + w - float(row[tid2pdf[il]]), dst, ol, words)
                for s, (cost, words) in toks.items() if cost <= weight_cutoff
                for dst, il, ol, w in out[s] if il != 0]
        new = {}
        if cand:
            next_cutoff = min(c[0] for c in cand) + beam
            for total, dst, ol, words in cand:
                if total > next_cutoff:
                    continue
                c = f32(total)
                if dst not in new or c < new[dst][0]:
                    new[dst] = (c, words + (ol,) if ol else words)
            close(new, f32(next_cutoff))
        toks = new
        yield toks


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["loop", "eps"])
def test_partials_follow_the_host_restatement(ctx, kind):
    am, fst, graph, tid2pdf = make_model(ctx, kind)
    pcms = [coloured(200 + u, n) for u, n in enumerate(LENS)]
    _, _, rows = batch_rows(ctx, am, fst, pcms)
    per_frame = [[dict(t) for t in host_frames(graph, tid2pdf, r)] for r in rows]
    T = [r.shape[0] for r in rows]
    dec = pk.Decoder(ctx, am, fst, len(rows))
    checked = [0]

    def each(t):
        words, cost, frames = dec.partial()
        for s in range(len(rows)):
            n = min(t, T[s])
            assert frames[s] == n
            if n == 0:
                continue
            toks = per_frame[s][n - 1]
            c, st = min((c, st) for st, (c, _) in toks.items())
            assert words[s] == list(toks[st][1]), (s, t)
            assert abs(cost[s] - c) <= 1e-5 * max(1.0, abs(c)), (s, t, cost[s], c)
            checked[0] += 1

    decode_in_splits(dec, rows, 7, each)
    assert checked[0] > 50
    words, cost, frames = dec.partial()
    assert np.all(frames == 0)   # finished: fresh utterances
    dec.close()


# ---------------------------------------------------------------- attached to a stream
def stream_utterance(st, dec, ref, pcm, chunk, rows=True):
    """Pushes pcm [S][n] chunk by chunk; the host-fed `ref` decoder gets the rows the stream returns
    and must agree bitwise after every push. Returns the decoder's finish() (None without one), its
    best-so-far after every call and how many pushes and flushes emitted frames."""
    buf = np.empty((pcm.shape[0], chunk), np.int16)
    parts, emitting = [], 0
    frames = lambda o: o.shape[1] if rows else o
    for k in range(pcm.shape[1] // chunk):
        buf[:] = pcm[:, k * chunk:(k + 1) * chunk]
        o = st.push(buf, rows=rows)
        emitting += frames(o) > 0
        if dec is None:
            continue
        if ref is not None and rows and o.shape[1]:
            ref.advance(o)
        parts.append(dec.partial())
        if ref is not None:
            r = ref.partial()
            assert parts[-1][0] == r[0] and np.array_equal(parts[-1][1], r[1]) and np.array_equal(parts[-1][2], r[2])
    o = st.flush(rows=rows)
    emitting += frames(o) > 0
    if dec is None:
        return None, parts, emitting
    if ref is not None and rows and o.shape[1]:
        ref.advance(o)
    parts.append(dec.partial())
    got = dec.finish()
    if ref is not None:
        want = ref.finish()
        assert got[0] == want[0] and np.array_equal(got[1], want[1])
    return got, parts, emitting


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["loop", "eps"])
@pytest.mark.parametrize("chunk", [160, 2560, 16000])
def test_attached_stream_decodes_like_the_batch(ctx, kind, chunk):
    am, fst, _, _ = make_model(ctx, kind)
    S, n = 5, 64000   # a multiple of every chunk size
    g = synth_global_cmvn()
    st = pk.Stream(ctx, am, S, chunk, g, 0.1)
    dec = pk.Decoder(ctx, am, fst, S)
    ref = pk.Decoder(ctx, am, fst, S)
    st.set_decoder(dec)
    for rep in range(2):   # a second utterance through the same objects
        pcm = np.stack([coloured(300 + 10 * rep + s, n) for s in range(S)])
        (hyps, wts), _, _ = stream_utterance(st, dec, ref, pcm, chunk)
        bh, bw, rows = batch_rows(ctx, am, fst, list(pcm))
        assert hyps == bh, (rep, hyps, bh)
        for s in range(S):
            T = rows[s].shape[0]
            assert abs(wts[s] / T - bw[s] / T) < 2e-3
    st.close()
    dec.close()
    ref.close()


def check_decode_only_pushes():
    ctx = pk.Context(0)
    am, fst, _, _ = make_model(ctx, "loop")
    S, chunk, n_chunks = 4, 2560, 14
    pcm = np.stack([coloured(400 + s, chunk * n_chunks) for s in range(S)])
    st = pk.Stream(ctx, am, S, chunk, synth_global_cmvn(), 0.1)
    dec = pk.Decoder(ctx, am, fst, S)
    misc = lambda: ctx.profile_get()["misc"][0]
    # the same utterance without a decoder: the stream's own launches of the misc class (counted on
    # a second utterance, which follows a flush like every utterance below)
    stream_utterance(st, None, None, pcm, chunk, rows=True)
    m0 = misc()
    _, _, emitting = stream_utterance(st, None, None, pcm, chunk, rows=True)
    bare = misc() - m0
    assert emitting == n_chunks + 1
    st.set_decoder(dec)
    r0, m0 = st.graph_replays(), misc()
    full, parts_full, _ = stream_utterance(st, dec, None, pcm, chunk, rows=True)
    m1 = misc()
    only, parts_only, _ = stream_utterance(st, dec, None, pcm, chunk, rows=False)
    # exactly one advance per push or flush that emits frames, replays included, and the finish
    assert m1 - m0 == bare + emitting + 1
    assert misc() - m1 == bare + emitting + 1
    # from the fourth push on (the first three differ in carried tail and context rows; then the
    # shapes and the host buffers stay the same) every push replays a captured graph
    replays = st.graph_replays() - r0
    if os.environ.get("PKB_STREAM_GRAPH") == "0":
        assert replays == 0
    else:
        assert replays == 2 * (n_chunks - 3), replays
    assert full[0] == only[0] and np.array_equal(full[1], only[1])
    assert all(len(h) > 0 for h in full[0])
    for a, b in zip(parts_full, parts_only):
        assert a[0] == b[0] and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
    # the same utterance, rows returned, through a host-fed decoder
    ref = pk.Decoder(ctx, am, fst, S)
    again, _, _ = stream_utterance(st, dec, ref, pcm, chunk, rows=True)
    assert again[0] == full[0] and np.array_equal(again[1], full[1])
    for o in (st, dec, ref):
        o.close()
    ctx.close()


@pytest.mark.gpu
def test_decode_only_pushes_in_the_captured_graph():
    check_decode_only_pushes()


@pytest.mark.gpu
def test_decode_only_pushes_eager():
    run_child("import test_gpu_online_decode as t\nt.check_decode_only_pushes()\nprint('CHILD OK')",
              PKB_STREAM_GRAPH="0")


# ---------------------------------------------------------------- record compaction
def one_word_rows(P, n_hmm_states, word, T):
    """Rows of demo.word_loop_graph's pdf layout on which only `word` survives the beam: its state
    s's pdf scores 0 for a third of the frames each, every other pdf -1000."""
    stride = max(1, P // n_hmm_states)
    rows = np.full((T, P), -1000.0, np.float32)
    for t in range(T):
        rows[t, (word * 3 + min(3 * t // T, 2)) * stride] = 0.0
    return rows



def host_record_counts(graph, tid2pdf, loglik, every, beam=16.0):
    """The host restatement with word records as decoder.cu keeps them: one record per token whose
    winning arc carries an output label, per frame. Returns (records appended, largest number of
    records reachable from the live tokens at an advance boundary, most records appended by one
    advance)."""
    num_states, start, finals, arcs = graph
    assert all(il != 0 for _, _, il, _, _ in arcs)   # a graph without epsilon arcs
    out = [[] for _ in range(num_states)]
    for src, dst, il, ol, w in arcs:
        out[src].append((dst, il, ol, float(np.float32(w))))
    prev = []
    toks = {start: (0.0, -1)}
    appended, live_max, adv_max, adv = 0, 0, 0, 0
    for t, row in enumerate(loglik):
        weight_cutoff = float(np.float32(min(c for c, _ in toks.values()) + beam))
        cand = [(cost + w - float(row[tid2pdf[il]]), dst, ol, rec)
                for s, (cost, rec) in toks.items() if cost <= weight_cutoff
                for dst, il, ol, w in out[s]]
        next_cutoff = min(c[0] for c in cand) + beam
        win = {}
        for total, dst, ol, rec in cand:
            if total <= next_cutoff:
                c = float(np.float32(total))
                if dst not in win or c < win[dst][0]:
                    win[dst] = (c, ol, rec)
        toks = {}
        for dst, (c, ol, rec) in win.items():
            if ol:
                prev.append(rec)
                rec = len(prev) - 1
                appended += 1
                adv += 1
            toks[dst] = (c, rec)
        if (t + 1) % every == 0 or t + 1 == len(loglik):
            seen = set()
            for _, rec in toks.values():
                while rec >= 0 and rec not in seen:
                    seen.add(rec)
                    rec = prev[rec]
            live_max = max(live_max, len(seen))
            adv_max = max(adv_max, adv)
            adv = 0
    return appended, live_max, adv_max


@pytest.mark.gpu
def test_record_compaction_on_a_long_stream(ctx):
    am, fst, graph, tid2pdf = make_model(ctx, "loop")
    pcm = coloured(500, 120 * 16000)
    hyps, wts, rows = batch_rows(ctx, am, fst, [pcm])
    every = 16
    appended, live_max, adv_max = host_record_counts(graph, tid2pdf, rows[0], every)
    max_records = max(2 * live_max, 2 * adv_max)
    assert max_records <= appended // 4, (max_records, appended)
    res = []
    for mr in (0, max_records):
        dec = pk.Decoder(ctx, am, fst, 1, max_records=mr)
        res.append(decode_in_splits(dec, rows, every))
        dec.close()
    (h0, w0), (h1, w1) = res
    assert h0[0] is not None and h1[0] is not None
    assert h0 == h1 == hyps
    assert np.array_equal(w0.view(np.int32), w1.view(np.int32)) and np.array_equal(w0, wts)
    assert len(hyps[0]) > 16

    # a store smaller than the surviving history is reported, and the decoder recovers
    dec = pk.Decoder(ctx, am, fst, 1, max_records=16)
    seen_neg = []
    h, _ = decode_in_splits(dec, rows, every, lambda t: seen_neg.append(dec.partial()[0][0] is None))
    assert h == [None] and any(seen_neg)
    h, w = decode_in_splits(dec, [one_word_rows(am.num_pdfs(), 36, 5, 60)], every)
    want, ww = host_viterbi(graph, tid2pdf, one_word_rows(am.num_pdfs(), 36, 5, 60))
    assert h == [want] and want == [6]
    assert abs(w[0] - ww) <= 1e-6 * abs(ww)
    dec.close()


# ---------------------------------------------------------------- errors and lifetime
@pytest.mark.gpu
def test_invalid_uses_are_rejected(ctx):
    am, fst, graph, tid2pdf = make_model(ctx, "loop")
    g = synth_global_cmvn()
    S, chunk = 3, 2560
    st = pk.Stream(ctx, am, S, chunk, g, 0.1)
    dec = pk.Decoder(ctx, am, fst, S)
    # compact output and a decoder exclude each other
    st.set_compact(True)
    with pytest.raises(pk.PkbError):
        st.set_decoder(dec)
    st.set_compact(False)
    st.set_decoder(dec)
    with pytest.raises(pk.PkbError):
        st.set_compact(True)
    # another stream count, another model, another context
    other = pk.Decoder(ctx, am, fst, S + 1)
    st2 = pk.Stream(ctx, am, S + 1, chunk, g, 0.1)
    with pytest.raises(pk.PkbError):
        st2.set_decoder(dec)
    am2, fst2, _, _ = make_model(ctx, "loop")
    dec2 = pk.Decoder(ctx, am2, fst2, S)
    st5 = pk.Stream(ctx, am, S, chunk, g, 0.1)
    with pytest.raises(pk.PkbError):
        st5.set_decoder(dec2)
    ctx2 = pk.Context(0)
    am3, fst3, _, _ = make_model(ctx2, "loop")
    dec3 = pk.Decoder(ctx2, am3, fst3, S)
    st3 = pk.Stream(ctx, am, S, chunk, g, 0.1)
    with pytest.raises(pk.PkbError):
        st3.set_decoder(dec3)
    with pytest.raises(pk.PkbError):     # FST of another context
        pk.Decoder(ctx, am, fst3, S)
    # a push after the flush before the decoder is finished
    pcm = np.stack([coloured(600 + s, chunk) for s in range(S)])
    st.push(pcm, rows=False)
    st.flush(rows=False)
    with pytest.raises(pk.PkbError):
        st.push(pcm, rows=False)
    dec.finish()
    st.push(pcm, rows=False)
    # more frames than the stride
    with pytest.raises(pk.PkbError):
        other.advance(np.zeros((S + 1, 4, am.num_pdfs()), np.float32), [5] * (S + 1))
    # destroying the decoder detaches it; destroying a stream leaves its decoder usable
    st.flush(rows=False)
    dec.finish()
    dec.close()
    assert st.push(pcm).shape[0] == S      # rows only, nothing attached
    st.flush()
    st2.close()
    st4 = pk.Stream(ctx, am, S + 1, chunk, g, 0.1)
    st4.set_decoder(other)
    st4.close()
    other.advance(np.zeros((S + 1, 4, am.num_pdfs()), np.float32))
    words, _, frames = other.partial()
    assert np.all(frames == 4)
    for o in (other, dec2, dec3, st, st3, st5, fst2, am2, fst3, am3):
        o.close()
    ctx2.close()


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
    _, _, rows = batch_rows(ctx, am, fst, [synth_pcm(5, [0], 16000)[0], synth_pcm(5, [1], 16000)[0]])
    dec = pk.Decoder(ctx, am, fst, 2, max_tokens=64)
    hyps, _ = decode_in_splits(dec, rows, 16)
    assert hyps == [None, None]
    clean = one_word_rows(P, 600, 7, 30)
    hyps, wts = decode_in_splits(dec, [clean, clean], 16)
    want, ww = host_viterbi(graph, tid2pdf, clean)
    assert hyps == [want, want] and want == [8]
    assert np.allclose(wts, ww, rtol=1e-6)
    dec.close()
    fst.close()
    am.close()


@pytest.mark.gpu
def test_create_attach_finish_destroy_cycles_do_not_leak(ctx):
    import torch
    am, fst, _, _ = make_model(ctx, "loop")
    g = synth_global_cmvn()
    S, chunk = 4, 2560
    pcm = np.stack([coloured(700 + s, chunk) for s in range(S)])

    def cycle():
        st = pk.Stream(ctx, am, S, chunk, g, 0.1)
        dec = pk.Decoder(ctx, am, fst, S)
        st.set_decoder(dec)
        for _ in range(3):
            st.push(pcm, rows=False)
        st.flush(rows=False)
        dec.finish()
        dec.close()
        st.close()

    cycle()
    before = torch.cuda.mem_get_info(0)[0]
    for _ in range(20):
        cycle()
    assert before - torch.cuda.mem_get_info(0)[0] <= MARGIN
