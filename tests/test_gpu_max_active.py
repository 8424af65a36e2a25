"""Max-active pruning of the GPU search (pkb_batch_set_max_active, pkb_decoder_set_max_active): on a
frame of more than max_active tokens whose max_active-th smallest cost c_k is below float(best +
beam), only the tokens of cost <= c_k are expanded and the next bound adds float(min(beam, (c_k -
best) + 0.5)). Decode words and weights must equal a host restatement of the pruned decode (pinned to
oracle/decoder.host_viterbi without pruning), lattices a host restatement of the pruned lattice, bit
for bit, on every kernel path; the online decoder must equal the batch for any split, attached to a
stream too."""

import math
import os
import sys

import numpy as np
import pytest

import pocketkaldi_b200 as pk
import tools.decode_demo as demo
from oracle.decoder import host_viterbi as oracle_viterbi
from pocketkaldi_b200 import formats
from pocketkaldi_b200.synth import synth_global_cmvn

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from test_gpu_lattice import host_lattice, lattice_best_path, same_records, tiny_graph  # noqa: E402
from test_gpu_online_decode import decode_in_splits, run_child, stream_utterance  # noqa: E402
from test_gpu_viterbi import coloured, eps_graph  # noqa: E402

LENS = [16000, 24000, 8000, 32000, 400, 12345]
MARGIN = 64 << 20
LB = 4.0


# ---------------------------------------------------------------- host restatement
def host_viterbi(graph, tid2pdf, loglik, beam=16.0, max_active=0):
    """oracle/decoder.host_viterbi (the reference decoder's arithmetic) with the max-active rule:
    with more than max_active tokens whose max_active-th smallest cost c_k is below the weight
    cutoff, the cutoff becomes c_k and the next cutoff adds float(min(beam, (c_k - best) + 0.5))
    instead of beam. Returns (word ids, weight)."""
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
        best = min(c for c, _ in toks.values())
        weight_cutoff = f32(best + beam)
        adaptive = beam
        if 0 < max_active < len(toks):
            ck = sorted(c for c, _ in toks.values())[max_active - 1]
            if ck < weight_cutoff:
                weight_cutoff, adaptive = ck, f32(min(beam, (ck - best) + 0.5))
        cand = [(cost + w - float(row[tid2pdf[il]]), dst, ol, words)
                for s, (cost, words) in toks.items() if cost <= weight_cutoff
                for dst, il, ol, w in out[s] if il != 0]
        if not cand:
            return [], 0.0
        next_cutoff = min(c[0] for c in cand) + adaptive
        new = {}
        for total, dst, ol, words in cand:
            if total > next_cutoff:
                continue
            c = f32(total)
            if dst not in new or c < new[dst][0]:
                new[dst] = (c, words + (ol,) if ol else words)
        close(new, f32(next_cutoff))
        toks = new
    ends = [(f32(c + finals[s]), s, words) for s, (c, words) in toks.items() if s in finals]
    if not ends:
        return [], 0.0
    c, s, words = min(ends)
    return list(words), f32(c + finals[s])


def host_lattice_ma(graph, tid2pdf, loglik, beam=16.0, lattice_beam=8.0, max_active=0, stats=None):
    """test_gpu_lattice.host_lattice with the max-active rule in the weight cutoff and the next
    bound. stats (a list) receives per frame (live tokens, tokens expanded, c_k or None when the
    frame has at most max_active tokens, tokens of cost c_k)."""
    num_states, start, finals, arcs = graph
    arcs = sorted(arcs)
    S = num_states
    src = np.array([a[0] for a in arcs], np.int64)
    dst = np.array([a[1] for a in arcs], np.int64)
    il = np.array([a[2] for a in arcs], np.int64)
    ol = np.array([a[3] for a in arcs], np.int64)
    w = np.array([a[4] for a in arcs], np.float32).astype(np.float64)
    fin = np.full(S, np.inf)
    for s, v in finals.items():
        fin[s] = float(np.float32(v))
    eps = np.nonzero(il == 0)[0]
    emit = il != 0
    pdf = np.asarray(tid2pdf, np.int64)[il]
    beam = float(np.float32(beam))
    f32 = lambda x: np.asarray(x, np.float32).astype(np.float64)

    def close(alpha, cutoff):
        while True:
            a = alpha[src[eps]]
            tot = a + w[eps]
            ok = np.isfinite(a) & (tot <= cutoff)
            new = alpha.copy()
            np.minimum.at(new, dst[eps[ok]], f32(tot[ok]))
            if np.array_equal(new, alpha):
                return alpha
            alpha = new

    def eps_included(alpha, cutoff):
        a = alpha[src[eps]]
        return eps[np.isfinite(a) & (a + w[eps] <= cutoff)]

    empty = np.zeros(0, pk.LATTICE_ARC_DTYPE)
    alpha = np.full(S, np.inf)
    alpha[start] = 0.0
    alpha = close(alpha, np.inf)
    alphas, acs, g_eps, g_emit = [alpha], [], [eps_included(alpha, np.inf)], []
    for row in loglik:
        live = np.sort(alpha[np.isfinite(alpha)])
        best = float(live[0])
        wc = float(np.float32(best + beam))
        adaptive, ck = beam, None
        if 0 < max_active < len(live):
            ck = float(live[max_active - 1])
            if ck < wc:
                wc, adaptive = ck, float(np.float32(min(beam, (ck - best) + 0.5)))
        if stats is not None:
            stats.append((len(live), int((live <= wc).sum()), ck, int((live == ck).sum())))
        ac = -np.asarray(row, np.float32)[pdf].astype(np.float64)
        tot = (alpha[src] + w) + ac
        m = emit & (alpha[src] <= wc)
        if not m.any():
            return empty, math.inf, sum(len(g) for g in g_eps + g_emit)
        nc = tot[m].min() + adaptive
        keep = m & (tot <= nc)
        new = np.full(S, np.inf)
        np.minimum.at(new, dst[keep], f32(tot[keep]))
        cut = float(np.float32(nc))
        new = close(new, cut)
        acs.append(ac)
        g_emit.append(np.nonzero(keep)[0])
        g_eps.append(eps_included(new, cut))
        alphas.append(new)
        alpha = new
    T = len(acs)
    n_log = sum(len(g) for g in g_eps + g_emit)
    fa = alpha + fin
    best = float(fa[np.isfinite(fa)].min()) if np.isfinite(fa).any() else math.inf
    if best == math.inf:
        return empty, best, n_log
    bound = best + float(np.float32(lattice_beam))

    def eps_fix(beta, e):
        while True:
            new = beta.copy()
            np.minimum.at(new, src[e], w[e] + beta[dst[e]])
            if np.array_equal(new, beta):
                return beta
            beta = new

    kept_eps, kept_emit = [None] * (T + 1), [None] * T
    beta_next = None
    for t in range(T, -1, -1):
        if t == T:
            beta = fin.copy()
        else:
            e = g_emit[t]
            beta = np.full(S, np.inf)
            bh = beta_next[dst[e]]
            np.minimum.at(beta, src[e], (w[e] + acs[t][e]) + bh)
            lhs = ((alphas[t][src[e]] + w[e]) + acs[t][e]) + bh
            kept_emit[t] = e[np.isfinite(bh) & (lhs <= bound)]
        e = g_eps[t]
        beta = eps_fix(beta, e)
        bh = beta[dst[e]]
        lhs = ((alphas[t][src[e]] + w[e]) + 0.0) + bh
        kept_eps[t] = e[np.isfinite(bh) & (lhs <= bound)]
        beta_next = beta
    recs = []
    for t in range(T + 1):
        for e, ac in ((kept_eps[t], None), (kept_emit[t] if t < T else np.zeros(0, np.int64), t)):
            for a in e:
                recs.append((t, src[a], dst[a], il[a], ol[a], np.float32(w[a]),
                             np.float32(acs[ac][a]) if ac is not None else np.float32(0.0)))
    return np.array(recs, pk.LATTICE_ARC_DTYPE), best, n_log


def host_cases():
    """(graph, tid2pdf, loglik) of tiny random graphs and small word loops, in flat and peaked rows."""
    for seed in range(10):
        rng = np.random.default_rng(500 + seed)
        graph, tid2pdf = demo.word_loop_graph(6, 3, 24) if seed % 2 else tiny_graph(rng, 8)
        P = max(tid2pdf) + 1
        T = int(rng.integers(5, 40))
        loglik = rng.uniform(-6.0 if seed % 3 else -1.0, 0.0, (T, P)).astype(np.float32)
        yield seed, graph, tid2pdf, loglik


# ---------------------------------------------------------------- CPU: the restatement itself
def test_decode_restatement_at_zero_is_the_oracle():
    for seed, graph, tid2pdf, loglik in host_cases():
        assert host_viterbi(graph, tid2pdf, loglik) == oracle_viterbi(graph, tid2pdf, loglik), seed


def test_restatement_at_zero_is_the_lattice_restatement():
    for seed, graph, tid2pdf, loglik in host_cases():
        for lb in (0.5, LB, math.inf):
            got = host_lattice_ma(graph, tid2pdf, loglik, lattice_beam=lb)
            want = host_lattice(graph, tid2pdf, loglik, lattice_beam=lb)
            assert same_records(got[0], want[0]) and got[1:] == want[1:], (seed, lb)


def test_no_frame_expands_more_than_max_active_plus_the_ties():
    pruned = 0
    for seed, graph, tid2pdf, loglik in host_cases():
        for ma in (1, 2, 4, 8):
            stats = []
            words, _ = host_viterbi(graph, tid2pdf, loglik, max_active=ma)
            lat, _, _ = host_lattice_ma(graph, tid2pdf, loglik, lattice_beam=LB, max_active=ma, stats=stats)
            for n, expanded, ck, ties in stats:
                assert 1 <= expanded <= n
                if ck is None:
                    assert n <= ma
                    continue
                # fewer than max_active tokens cost less than c_k; every tie at c_k is expanded too
                assert expanded <= ma - 1 + ties, (seed, ma, n, expanded, ties)
                pruned += expanded < n
            # the best path through the pruned lattice is the pruned decode
            bp = lattice_best_path(lat, len(loglik), graph[1], graph[2])
            assert (bp is None and words == []) or bp[0] == words, (seed, ma)
    assert pruned > 20


def test_max_active_of_the_state_count_is_the_unpruned_search():
    for seed, graph, tid2pdf, loglik in host_cases():
        S = graph[0]
        w0 = host_viterbi(graph, tid2pdf, loglik)
        l0 = host_lattice_ma(graph, tid2pdf, loglik, lattice_beam=LB)
        for ma in (S, S + 1, 10 ** 6):
            assert host_viterbi(graph, tid2pdf, loglik, max_active=ma) == w0, (seed, ma)
            got = host_lattice_ma(graph, tid2pdf, loglik, lattice_beam=LB, max_active=ma)
            assert same_records(got[0], l0[0]) and got[1:] == l0[1:], (seed, ma)


def test_pruning_changes_words_on_flat_rows():
    # teeth for the restatement: on flat acoustic rows a max_active of 1 follows a greedy path
    changed = 0
    for seed in range(6):
        rng = np.random.default_rng(900 + seed)
        graph, tid2pdf = demo.word_loop_graph(6, 3, 24)
        loglik = rng.uniform(-1.0, 0.0, (60, 24)).astype(np.float32)
        changed += host_viterbi(graph, tid2pdf, loglik, max_active=1) != host_viterbi(graph, tid2pdf, loglik)
    assert changed > 0


# ---------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def ctx():
    c = pk.Context(0)
    yield c
    c.close()


KINDS = ["loop", "eps", "loop_mid", "loop_big"]


def make_model(ctx, kind):
    """The graphs of test_gpu_online_decode.make_model (dense kernel: "loop" 12 words, "eps" the
    epsilon hub; table kernel: "loop_mid" 301 states with shared-memory tables, "loop_big" 541
    states with global tables) under a network whose scores are left flat enough that many tokens
    stay inside the beam, so that max-active has something to prune."""
    rng = np.random.default_rng({"loop": 11, "eps": 12, "loop_big": 13, "loop_mid": 14}[kind])
    P = 600 if kind in ("loop_big", "loop_mid") else 96
    layers = formats.make_dnn(rng, 440, 96, 2, P)
    prior = rng.uniform(0.5, 1.5, P).astype(np.float32)
    prior /= prior.sum()
    if kind == "eps":
        graph, tid2pdf = eps_graph(10, 3, P)
    else:
        graph, tid2pdf = demo.word_loop_graph({"loop": 12, "loop_big": 180, "loop_mid": 100}[kind], 3, P)
    am = pk.AcousticModel(ctx, pk.PREC_BF16X3).from_layers(layers, prior, 5, 5, tid2pdf=tid2pdf)
    fst = pk.Fst(ctx, graph=graph)
    return am, fst, graph, tid2pdf


def batch_of(ctx, am, lens, seed=100):
    pcms = [coloured(seed + u, n) if n else np.zeros(0, np.int16) for u, n in enumerate(lens)]
    b = pk.Batch(ctx, lens, synth_global_cmvn(), am, prob_scale=0.1)
    if sum(lens):
        b.set_pcm(np.ascontiguousarray(np.concatenate(pcms), np.int16))
    b.run(pk.STAGE_ALL)
    ll = b.get(pk.BUF_LOGLIK)
    off = np.concatenate([[0], np.cumsum(b.num_frames)])
    return b, [ll[off[u]:off[u + 1]].copy() for u in range(len(lens))]


def same_lattices(a, b):
    return all(same_records(x, y) for x, y in zip(a[0], b[0])) and a[1].tobytes() == b[1].tobytes()


def values(graph):
    return (1, 16, 64, graph[0] + 1)


def test_graph_kinds_cover_every_kernel_path():
    # plan_viterbi (decoder.cu): dense up to 2048 states and 4096 arcs, then shared-memory tables up
    # to 512 states, global tables above
    for kind, want in (("loop", "dense"), ("loop_mid", "shared"), ("loop_big", "global")):
        ns, _, _, arcs = demo.word_loop_graph({"loop": 12, "loop_big": 180, "loop_mid": 100}[kind], 3, 600)[0]
        dense = ns <= 2048 and len(arcs) <= 4096
        assert ("dense" if dense else "shared" if ns <= 512 else "global") == want
    assert eps_graph(10, 3, 96)[0][0] <= 2048


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_batch_decode_and_lattice_equal_the_restatement_bitwise(ctx, kind):
    am, fst, graph, tid2pdf = make_model(ctx, kind)
    b, rows = batch_of(ctx, am, LENS + [0])
    for ma in values(graph):
        b.set_max_active(ma)
        hyps, wts = b.decode(fst)
        lats, best = b.lattice(fst, lattice_beam=LB)
        for u, r in enumerate(rows):
            want, wbest, _ = host_lattice_ma(graph, tid2pdf, r, lattice_beam=LB, max_active=ma)
            if ma <= 64:
                words, weight = host_viterbi(graph, tid2pdf, r, max_active=ma)
            else:
                # host_viterbi expands every token in Python; the restatement's lattice gives the
                # same words and weight (pinned on the CPU) at a fraction of the cost
                bp = lattice_best_path(want, r.shape[0], graph[1], graph[2])
                words, weight = ([], 0.0) if bp is None else (bp[0], np.float32(wbest) + np.float32(graph[2][bp[1]]))
            assert hyps[u] == words, (kind, ma, u)
            assert np.float32(wts[u]).tobytes() == np.float32(weight).tobytes(), (kind, ma, u, wts[u], weight)
            assert lats[u] is not None, (kind, ma, u)
            assert same_records(lats[u], want), (kind, ma, u, len(lats[u]), len(want))
            assert np.float64(best[u]).tobytes() == np.float64(wbest).tobytes(), (kind, ma, u)
    for o in (b, fst, am):
        o.close()


@pytest.mark.gpu
def test_pruning_changes_words_on_some_graph(ctx):
    changed = 0
    for kind in KINDS:
        am, fst, graph, _ = make_model(ctx, kind)
        b, _ = batch_of(ctx, am, LENS, seed=200)
        full, _ = b.decode(fst)
        b.set_max_active(1)
        pruned, _ = b.decode(fst)
        changed += sum(x != y for x, y in zip(full, pruned))
        for o in (b, fst, am):
            o.close()
    assert changed > 0


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_inactive_limits_change_nothing(ctx, kind):
    am, fst, graph, _ = make_model(ctx, kind)
    b, _ = batch_of(ctx, am, LENS, seed=300)
    hyps, wts = b.decode(fst)
    lat = b.lattice(fst, lattice_beam=LB)
    for ma in (graph[0], graph[0] + 1, 1 << 30, 0):
        b.set_max_active(ma)
        h, w = b.decode(fst)
        assert h == hyps and w.tobytes() == wts.tobytes(), (kind, ma)
        assert same_lattices(b.lattice(fst, lattice_beam=LB), lat), (kind, ma)
    for o in (b, fst, am):
        o.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_downstream_of_pruned_lattices(ctx, kind):
    am, fst, graph, _ = make_model(ctx, kind)
    b, rows = batch_of(ctx, am, LENS, seed=400)
    finals = graph[2]
    for ma in (1, 16):
        b.set_max_active(ma)
        hyps, wts = b.decode(fst)
        lats, best = b.lattice(fst, lattice_beam=LB)
        nb = b.nbest(fst, n=5)
        _, arc_post, _ = b.posteriors(fst)
        for u, r in enumerate(rows):
            bp = lattice_best_path(lats[u], r.shape[0], graph[1], finals)
            if bp is None:
                assert hyps[u] == [] and best[u] == math.inf and nb[u] == []
                continue
            words, s, c = bp
            assert words == hyps[u], (kind, ma, u)
            assert np.float32(np.float32(best[u]) + np.float32(finals[s])) == wts[u]
            assert nb[u][0][0] == hyps[u], (kind, ma, u)
            lat = lats[u]
            T = int(lat["t"][lat["ilabel"] != 0].max()) + 1
            for t in range(T):
                m = (lat["t"] == t) & (lat["ilabel"] != 0)
                assert abs(float(arc_post[u][m].astype(np.float64).sum()) - 1.0) < 1e-4, (kind, ma, u, t)
    for o in (b, fst, am):
        o.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_online_splits_equal_the_batch_bitwise(ctx, kind):
    am, fst, graph, _ = make_model(ctx, kind)
    b, rows = batch_of(ctx, am, LENS, seed=500)
    for ma in (1, 16):
        b.set_max_active(ma)
        hyps, wts = b.decode(fst)
        lat = b.lattice(fst, lattice_beam=LB)
        for lattices in (False, True):
            for k in (1, 7, 16, max(r.shape[0] for r in rows)):
                dec = pk.Decoder(ctx, am, fst, len(rows))
                dec.set_max_active(ma)
                if lattices:
                    dec.set_lattice(LB)
                got, gw = decode_in_splits(dec, rows, k)
                assert got == hyps and gw.tobytes() == wts.tobytes(), (kind, ma, lattices, k)
                if lattices:
                    assert same_lattices(dec.lattice(), lat), (kind, ma, k)
                dec.close()
    for o in (b, fst, am):
        o.close()


def check_attached_stream():
    """A decoder attached to a stream, with max_active changed between utterances, against a
    host-fed decoder over the rows the stream returns (stream_utterance compares every partial and
    the finish); lattices on, so that the pushes carry the lattice work too."""
    ctx = pk.Context(0)
    am, fst, graph, tid2pdf = make_model(ctx, "loop")
    S, chunk, n = 4, 2560, 2560 * 12
    st = pk.Stream(ctx, am, S, chunk, synth_global_cmvn(), 0.1)
    dec = pk.Decoder(ctx, am, fst, S)
    dec.set_lattice(LB)
    st.set_decoder(dec)
    graphs = os.environ.get("PKB_STREAM_GRAPH") != "0"
    seen = {}
    for rep, ma in enumerate((16, 1, 0, 1)):
        dec.set_max_active(ma)
        ref = pk.Decoder(ctx, am, fst, S)
        ref.set_max_active(ma)
        ref.set_lattice(LB)
        pcm = np.stack([coloured(600 + s, n) for s in range(S)])   # the same audio every time
        r0 = st.graph_replays()
        (hyps, wts), parts, _ = stream_utterance(st, dec, ref, pcm, chunk)
        assert (st.graph_replays() > r0) == graphs, (rep, ma)
        lat = dec.lattice()
        assert same_lattices(lat, ref.lattice()), (rep, ma)
        key = ([h for h in hyps], wts.tobytes(), [(p[0], p[1].tobytes()) for p in parts])
        if ma in seen:
            assert key == seen[ma], ma
        seen[ma] = key
        ref.close()
    # the values give different searches, so the checks above see which value each pass used
    assert seen[1] != seen[0]
    with pytest.raises(pk.PkbError):
        dec.set_max_active(-1)
    for o in (st, dec, fst, am):
        o.close()
    ctx.close()


@pytest.mark.gpu
def test_attached_stream_follows_max_active():
    check_attached_stream()


@pytest.mark.gpu
def test_attached_stream_follows_max_active_eager():
    run_child("import test_gpu_max_active as t\nt.check_attached_stream()\nprint('CHILD OK')",
              PKB_STREAM_GRAPH="0")


@pytest.mark.gpu
def test_invalid_uses_are_rejected_and_the_setting_persists(ctx):
    am, fst, graph, tid2pdf = make_model(ctx, "loop")
    b, rows = batch_of(ctx, am, LENS[:3], seed=700)
    with pytest.raises(pk.PkbError):
        b.set_max_active(-1)
    b.set_max_active(1)
    with pytest.raises(pk.PkbError):
        b.set_max_active(-5)          # a rejected value leaves the setting alone
    for _ in range(2):
        hyps, wts = b.decode(fst)
        for u, r in enumerate(rows):
            words, weight = host_viterbi(graph, tid2pdf, r, max_active=1)
            assert hyps[u] == words and np.float32(wts[u]) == np.float32(weight)
        b.lattice(fst, lattice_beam=LB)
    dec = pk.Decoder(ctx, am, fst, 2)
    with pytest.raises(pk.PkbError):
        dec.set_max_active(-1)
    dec.set_max_active(4)
    dec.advance(np.zeros((2, 3, am.num_pdfs()), np.float32))
    with pytest.raises(pk.PkbError):
        dec.set_max_active(8)         # in the middle of an utterance
    dec.finish()
    dec.set_max_active(8)
    for o in (dec, b, fst, am):
        o.close()


@pytest.mark.gpu
def test_create_set_destroy_cycles_do_not_leak(ctx):
    import torch
    am, fst, _, _ = make_model(ctx, "loop_big")
    g = synth_global_cmvn()
    S, chunk = 3, 2560
    pcm = np.stack([coloured(800 + s, chunk) for s in range(S)])

    def cycle():
        b, _ = batch_of(ctx, am, [chunk] * 2, seed=800)
        b.set_max_active(16)
        b.decode(fst)
        b.lattice(fst, lattice_beam=LB)
        b.close()
        st = pk.Stream(ctx, am, S, chunk, g, 0.1)
        dec = pk.Decoder(ctx, am, fst, S)
        dec.set_max_active(16)
        st.set_decoder(dec)
        for _ in range(5):
            st.push(pcm, rows=False)
        st.flush(rows=False)
        dec.finish()
        dec.set_max_active(0)
        dec.close()
        st.close()

    cycle()
    before = torch.cuda.mem_get_info(0)[0]
    for _ in range(20):
        cycle()
    assert before - torch.cuda.mem_get_info(0)[0] <= MARGIN
    fst.close()
    am.close()
