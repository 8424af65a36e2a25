"""Best paths with frame alignments over lattices (pkb_batch_best_path, pkb_decoder_best_path): the
GPU results must equal, bit for bit, a host restatement of the tropical forward pass and traceback in
the fold order of include/pkb200.h; that restatement is pinned to brute-force enumeration of lattice
paths on tiny graphs."""

import math
import os
import sys

import numpy as np
import pytest

import pocketkaldi_b200 as pk
from pocketkaldi_b200.synth import synth_global_cmvn

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from test_gpu_lattice import LENS, batch_of, brute_force, host_lattice, same_records, tiny_graph  # noqa: E402
from test_gpu_nbest import key as nbest_key, lattice_T  # noqa: E402
from test_gpu_online_decode import MARGIN, decode_in_splits, make_model, run_child  # noqa: E402
from test_gpu_online_lattice import stream_rows  # noqa: E402
from test_gpu_posteriors import bits as post_bits, eps_cycle_model, fst_states  # noqa: E402
from test_gpu_viterbi import coloured  # noqa: E402

INF = math.inf
# (acoustic_scale, graph_scale, word_penalty): the search's own costs, a rescaled pair, an LMWT-style
# scale with a negative penalty and one with a positive penalty
TRIPLES = [(1.0, 1.0, 0.0), (0.3, 1.5, 0.0), (1.0 / 12, 1.0, -2.5), (0.1, 1.0, 1.5)]


# ---------------------------------------------------------------- host restatement
def record_costs(lat, acoustic_scale, graph_scale, word_penalty):
    """c(r) of include/pkb200.h in double: graph_scale x graph + acoustic_scale x acoustic, plus the
    penalty on a word."""
    as_, gs, wp = (float(np.float32(x)) for x in (acoustic_scale, graph_scale, word_penalty))
    c = gs * lat["graph_cost"].astype(np.float64) + as_ * lat["acoustic_cost"].astype(np.float64)
    return np.where(lat["olabel"] != 0, c + wp, c)


def host_best_path(lat, T, start, finals, acoustic_scale=1.0, graph_scale=1.0, word_penalty=0.0,
                   num_states=None):
    """The tropical forward pass of include/pkb200.h in its fold order: a node takes the emitting
    records into it from time t - 1, then the epsilon records of time t (in Kahn levels), each in
    record order, and a candidate replaces the held value only when strictly smaller. Returns
    (cost, graph_cost, acoustic_cost, words, word_t, alignment, path records), or -8 for an
    epsilon cycle."""
    S = num_states or (max([start] + list(finals) + [int(x) for x in lat["src"]] +
                           [int(x) for x in lat["dst"]]) + 1)
    gs = float(np.float32(graph_scale))
    t_, src, dst = lat["t"].astype(np.int64), lat["src"].astype(np.int64), lat["dst"].astype(np.int64)
    emit = lat["ilabel"] != 0
    c = record_costs(lat, acoustic_scale, graph_scale, word_penalty)
    bounds = np.searchsorted(2 * t_ + emit, np.arange(2 * T + 3))

    def fold(held, win, Xsrc, recs):
        # per destination the least candidate, the first in record order among equal ones; it
        # replaces the held value only when strictly smaller
        if len(recs) == 0:
            return
        cand = Xsrc[src[recs]] + c[recs]
        d = dst[recs]
        order = np.lexsort((recs, cand, d))
        first = order[np.r_[True, np.diff(d[order]) != 0]]
        better = cand[first] < held[d[first]]
        held[d[first][better]] = cand[first][better]
        win[d[first][better]] = recs[first][better]

    X = np.full(S, INF)
    X[start] = 0.0
    win = np.full(S, -1)
    wins = []
    for t in range(T + 1):
        E = np.arange(bounds[2 * t], bounds[2 * t + 1])
        done = np.ones(S, bool)
        done[dst[E]] = False
        while not done.all():
            inc_ok = np.ones(S, bool)
            np.logical_and.at(inc_ok, dst[E], done[src[E]])
            ready = ~done & inc_ok
            if not ready.any():
                return -8
            fold(X, win, X, E[ready[dst[E]]])
            done |= ready
        wins.append(win)
        if t == T:
            break
        Y = np.full(S, INF)
        win = np.full(S, -1)
        fold(Y, win, X, np.arange(bounds[2 * t + 1], bounds[2 * t + 2]))
        X = Y
    cost, fs = INF, -1
    for s in sorted(finals):
        v = X[s] + gs * float(np.float32(finals[s]))
        if v < cost:
            cost, fs = v, s
    if fs < 0:
        return INF, INF, INF, [], [], [], []
    path, t, s = [], T, fs
    while wins[t][s] >= 0:
        r = int(wins[t][s])
        path.append(r)
        s = int(src[r])
        t -= int(emit[r])
    assert (t, s) == (0, start)
    path.reverse()
    g = a = 0.0
    for r in path:
        g += float(lat["graph_cost"][r])
        a += float(lat["acoustic_cost"][r])
    g += float(np.float32(finals[fs]))
    words = [int(lat["olabel"][r]) for r in path if lat["olabel"][r]]
    word_t = [int(lat["t"][r]) for r in path if lat["olabel"][r]]
    ali = [int(lat["ilabel"][r]) for r in path if lat["ilabel"][r]]
    return float(cost), g, a, words, word_t, ali, path


def enumerate_best(lat, T, start, finals, acoustic_scale, graph_scale, word_penalty):
    """Every complete path of the lattice with its cost summed in path order: (least cost, the paths
    of that cost as record tuples)."""
    gs = float(np.float32(graph_scale))
    c = record_costs(lat, acoustic_scale, graph_scale, word_penalty)
    out = {}
    for i, r in enumerate(lat):
        out.setdefault((int(r["t"]), int(r["src"])), []).append(i)
    paths = []

    def walk(t, s, cost, used):
        if t == T and s in finals:
            paths.append((cost + gs * float(np.float32(finals[s])), used))
        for i in out.get((t, s), []):
            walk(t + (1 if lat["ilabel"][i] else 0), int(lat["dst"][i]), cost + float(c[i]), used + (i,))

    walk(0, start, 0.0, ())
    if not paths:
        return INF, set()
    lo = min(p[0] for p in paths)
    return lo, {p[1] for p in paths if p[0] == lo}


def recs(rows):
    return np.array(rows, pk.LATTICE_ARC_DTYPE)


# ---------------------------------------------------------------- CPU: the restatement itself
@pytest.mark.parametrize("seed", range(12))
def test_host_best_path_against_path_enumeration(seed):
    rng = np.random.default_rng(seed)
    graph, tid2pdf = tiny_graph(rng)
    T = int(rng.integers(1, 6))
    loglik = rng.uniform(-3.0, 0.0, (T, 3)).astype(np.float32)
    _, best = brute_force(graph, tid2pdf, loglik)
    for lb in (0.5, 2.0, INF):
        lat, hbest, _ = host_lattice(graph, tid2pdf, loglik, beam=1e4, lattice_beam=lb)
        if hbest == INF:
            assert len(lat) == 0 and best == INF
            continue
        for triple in TRIPLES:
            got = host_best_path(lat, lattice_T(lat), graph[1], graph[2], *triple, num_states=graph[0])
            want, paths = enumerate_best(lat, lattice_T(lat), graph[1], graph[2], *triple)
            cost, g, a, words, word_t, ali, path = got
            assert cost == want, (seed, lb, triple, cost, want)
            assert tuple(path) in paths, (seed, lb, triple)
            assert len(ali) == lattice_T(lat) == T
            assert words == [int(lat["olabel"][r]) for r in path if lat["olabel"][r]]
            assert word_t == sorted(word_t)


def test_exact_ties_follow_the_fold_order():
    # (t, src, dst, ilabel, olabel, graph_cost, acoustic_cost)
    # three emitting candidates of equal cost into (1, 3): the first in record order wins
    lat = recs([(0, 0, 1, 0, 5, 1.0, 0.0), (0, 0, 2, 0, 6, 1.0, 0.0),
                (0, 0, 3, 1, 7, 2.0, 0.0), (0, 1, 3, 2, 0, 1.0, 0.0), (0, 2, 3, 3, 0, 1.0, 0.0)])
    assert host_best_path(lat, 1, 0, {3: 0.0})[3:6] == ([7], [0], [1])
    # an emitting candidate into (1, 3) ties with an epsilon one of time 1: emitting records come first
    lat = recs([(0, 0, 1, 0, 5, 1.0, 0.0), (0, 0, 2, 1, 0, 1.0, 1.0), (0, 1, 3, 2, 0, 0.0, 1.0),
                (1, 2, 3, 0, 9, 0.0, 0.0)])
    assert host_best_path(lat, 1, 0, {3: 0.0})[3:6] == ([5], [0], [2])
    # epsilon candidates into one node in record order, whatever their Kahn level: the direct record
    # (level 1) and the one through state 1 (level 2) tie, and the direct one comes first
    lat = recs([(0, 0, 1, 0, 0, 1.0, 0.0), (0, 0, 2, 0, 5, 2.0, 0.0), (0, 1, 2, 0, 6, 1.0, 0.0),
                (0, 2, 3, 1, 0, 0.0, 2.0)])
    assert host_best_path(lat, 1, 0, {3: 0.0})[3:6] == ([5], [0], [1])
    # equal totals at two final states go to the lower state, whatever the record order
    lat = recs([(0, 0, 2, 1, 3, 1.0, 1.0), (0, 0, 1, 2, 4, 1.0, 1.0)])
    assert host_best_path(lat, 1, 0, {1: 0.0, 2: 0.0})[3:6] == ([4], [0], [2])
    # the final weight counts once in the graph cost, scaled in the cost
    lat = recs([(0, 0, 1, 1, 0, 1.0, 0.25)])
    assert host_best_path(lat, 1, 0, {1: 0.5}, 1.0, 2.0)[:3] == (3.25, 1.5, 0.25)


@pytest.mark.parametrize("seed", range(8))
def test_integer_costs_with_ties_pick_a_least_path(seed):
    rng = np.random.default_rng(40 + seed)
    graph, tid2pdf = tiny_graph(rng, 6)
    n, start, finals, arcs = graph
    graph = (n, start, {s: float(int(4 * f)) for s, f in finals.items()},
             [(a, d, i, o, float(int(3 * w))) for a, d, i, o, w in arcs])
    T = int(rng.integers(2, 6))
    loglik = -rng.integers(0, 3, (T, 3)).astype(np.float32)
    lat, best, _ = host_lattice(graph, tid2pdf, loglik, beam=1e4, lattice_beam=INF)
    if best == INF:
        return
    for triple in ((1.0, 1.0, 0.0), (1.0, 1.0, 1.0), (0.5, 2.0, -1.0)):
        got = host_best_path(lat, T, start, graph[2], *triple, num_states=n)
        want, paths = enumerate_best(lat, T, start, graph[2], *triple)
        assert got[0] == want and tuple(got[6]) in paths, (seed, triple)


@pytest.mark.parametrize("seed", range(8))
def test_a_higher_penalty_never_adds_words(seed):
    rng = np.random.default_rng(70 + seed)
    graph, tid2pdf = tiny_graph(rng, 6)
    T = int(rng.integers(2, 8))
    loglik = rng.uniform(-3.0, 0.0, (T, 3)).astype(np.float32)
    lat, best, _ = host_lattice(graph, tid2pdf, loglik, beam=1e4, lattice_beam=INF)
    if best == INF:
        return
    counts = [len(host_best_path(lat, T, graph[1], graph[2], 1.0, 1.0, wp, num_states=graph[0])[3])
              for wp in (-4.0, -1.0, -0.25, 0.0, 0.25, 1.0, 4.0)]
    assert counts == sorted(counts, reverse=True), (seed, counts)


def test_epsilon_cycles_give_minus_8():
    loop = recs([(0, 0, 1, 1, 3, 0.25, 1.5), (1, 1, 1, 0, 7, 0.5, 0.0)])
    assert host_best_path(loop, 1, 0, {1: 0.125}) == -8
    two = recs([(0, 0, 1, 1, 3, 0.25, 1.5), (1, 1, 2, 0, 0, 0.5, 0.0), (1, 2, 1, 0, 0, 0.5, 0.0)])
    assert host_best_path(two, 1, 0, {1: 0.125}) == -8
    assert host_best_path(two[:2], 1, 0, {1: 0.125, 2: 0.0})[3:6] == ([3], [0], [1])


# ---------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def ctx():
    c = pk.Context(0)
    yield c
    c.close()


def bits(res):
    """Comparable form of best_path() output, bit patterns included."""
    return [None if r is None else (np.array(r[:3], np.float64).tobytes(),) + tuple(x.tobytes() for x in r[3:])
            for r in res]


def check_against_host(got, lats, best, graph, triple, where):
    for u, lat in enumerate(lats):
        if lat is None:
            assert got[u] is None
            continue
        cost, g, a, words, word_t, ali = got[u]
        if best[u] == INF:
            assert (cost, g, a) == (INF, INF, INF) and len(words) == len(word_t) == len(ali) == 0
            continue
        w = host_best_path(lat, lattice_T(lat), graph[1], graph[2], *triple, num_states=graph[0])
        assert np.array([cost, g, a]).tobytes() == np.array(w[:3]).tobytes(), (where, u, (cost, g, a), w[:3])
        assert words.tolist() == w[3] and word_t.tolist() == w[4] and ali.tolist() == w[5], (where, u)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["loop", "eps", "loop_mid", "loop_big"])
@pytest.mark.parametrize("lb", [0.5, 4.0, INF])
def test_best_path_matches_the_host_restatement(ctx, kind, lb):
    am, fst, graph, tid2pdf = make_model(ctx, kind)
    b, rows = batch_of(ctx, am, LENS + [0])
    lats, best = b.lattice(fst, lattice_beam=lb)
    for triple in TRIPLES:
        check_against_host(b.best_path(fst, *triple), lats, best, graph, triple, (kind, lb, triple))
    for o in (b, fst, am):
        o.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["loop", "eps", "loop_big"])
def test_consistency_with_decode_nbest_and_the_rows(ctx, kind):
    am, fst, graph, tid2pdf = make_model(ctx, kind)
    b, rows = batch_of(ctx, am, LENS, seed=700)
    hyps, _ = b.decode(fst)
    _, best = b.lattice(fst, lattice_beam=4.0)
    nb = b.nbest(fst, n=2)
    checked = 0
    for triple in TRIPLES:
        got = b.best_path(fst, *triple)
        for u, r in enumerate(rows):
            cost, g, a, words, word_t, ali = got[u]
            if cost == INF:
                assert best[u] == INF
                continue
            assert len(ali) == r.shape[0], (kind, triple, u)
            # the path's acoustic cost is its rows' costs at the aligned pdfs, in frame order
            want = 0.0
            for t, tid in enumerate(ali.tolist()):
                want += float(np.float32(-r[t][tid2pdf[tid]]))
            assert a == want, (kind, triple, u, a, want)
            if triple == (1.0, 1.0, 0.0):
                assert abs(cost - (g + a)) <= 1e-9 * max(1.0, abs(cost))
                lst = nb[u]
                if len(lst) == 1 or sum(lst[1][1:]) > sum(lst[0][1:]) + 1e-6:
                    assert words.tolist() == hyps[u] == lst[0][0], (kind, u)
                    checked += 1
    assert checked > 0
    for o in (b, fst, am):
        o.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["loop", "eps", "loop_big"])
def test_repeated_calls_are_identical_and_change_nothing(ctx, kind):
    am, fst, _, _ = make_model(ctx, kind)
    b, rows = batch_of(ctx, am, LENS, seed=300)
    hyps, wts = b.decode(fst)
    lats, best = b.lattice(fst, lattice_beam=4.0)
    nb = nbest_key(b.nbest(fst, n=4))
    post = post_bits(b.posteriors(fst, 0.3, 1.5, 1e-3))
    first = bits(b.best_path(fst, 0.1, 1.0, -2.5))
    for _ in range(2):
        assert bits(b.best_path(fst, 0.1, 1.0, -2.5)) == first
    b.best_path(fst)
    # N-best and posterior calls leave the best-path results valid, and are left unchanged by them
    b.best_path(fst, 0.1, 1.0, -2.5)
    assert nbest_key(b.nbest(fst, n=4)) == nb
    assert post_bits(b.posteriors(fst, 0.3, 1.5, 1e-3)) == post
    nw = int(sum(len(r[3]) for r in b.best_path(fst, 0.1, 1.0, -2.5)))
    b.nbest(fst, n=4)
    b.posteriors(fst)
    words = np.zeros(max(nw, 1), np.int32)
    assert ctx.lib.pkb_batch_best_path_get(b.h, words.ctypes.data, None, None) == 0
    assert words[:nw].tolist() == [w for r in first for w in np.frombuffer(r[1], np.int32).tolist()]
    lats2, best2 = b.lattice(fst, lattice_beam=4.0)
    assert best2.tobytes() == best.tobytes() and all(same_records(x, y) for x, y in zip(lats, lats2))
    b.best_path(fst)
    hyps2, wts2 = b.decode(fst)
    assert hyps2 == hyps and wts2.tobytes() == wts.tobytes()
    for o in (b, fst, am):
        o.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["loop", "eps"])
def test_online_best_path_equals_batch_best_path_for_any_split(ctx, kind):
    am, fst, _, _ = make_model(ctx, kind)
    lens = LENS + [0]
    b, rows = batch_of(ctx, am, lens, seed=500)
    b.lattice(fst, lattice_beam=4.0)
    want = [bits(b.best_path(fst, *tr)) for tr in TRIPLES]
    b.close()
    T = max(r.shape[0] for r in rows)
    for k in (1, 7, 16, T):
        dec = pk.Decoder(ctx, am, fst, len(lens))
        dec.set_lattice(4.0, max_frames=T)
        with pytest.raises(pk.PkbError):
            dec.best_path()    # no finish yet
        decode_in_splits(dec, rows, k)
        assert [bits(dec.best_path(*tr)) for tr in TRIPLES] == want, (kind, k)
        dec.close()
    fst.close()
    am.close()


@pytest.mark.gpu
def test_max_active_lattices(ctx):
    am, fst, graph, _ = make_model(ctx, "loop_mid")
    b, rows = batch_of(ctx, am, LENS, seed=600)
    b.set_max_active(16)
    lats, best = b.lattice(fst, lattice_beam=4.0)
    got = b.best_path(fst, 0.1, 1.0, -2.5)
    check_against_host(got, lats, best, graph, (0.1, 1.0, -2.5), "max_active")
    b.close()
    dec = pk.Decoder(ctx, am, fst, len(rows))
    dec.set_max_active(16)
    dec.set_lattice(4.0, max_frames=max(r.shape[0] for r in rows))
    decode_in_splits(dec, rows, 7)
    assert bits(dec.best_path(0.1, 1.0, -2.5)) == bits(got)
    for o in (dec, fst, am):
        o.close()


def check_attached_stream_best_path():
    ctx = pk.Context(0)
    am, fst, _, _ = make_model(ctx, "loop")
    S, n, chunk = 3, 32000, 2560
    st = pk.Stream(ctx, am, S, chunk, synth_global_cmvn(), 0.1)
    dec = pk.Decoder(ctx, am, fst, S)
    dec.set_lattice(4.0)
    st.set_decoder(dec)
    ref = pk.Decoder(ctx, am, fst, S)
    ref.set_lattice(4.0)
    for rep in range(2):
        pcm = np.stack([coloured(930 + 10 * rep + s, n) for s in range(S)])
        stream_rows(st, pcm, chunk, rows=False)   # decode-only pushes
        dec.finish()
        got = bits(dec.best_path(0.1, 1.0, -2.5))
        rows = stream_rows(st, pcm, chunk, rows=True)
        dec.finish()
        ref.advance(np.stack(rows))
        ref.finish()
        assert got == bits(ref.best_path(0.1, 1.0, -2.5)) == bits(dec.best_path(0.1, 1.0, -2.5)), rep
        res = dec.best_path()
        assert all(len(r[5]) == len(rows[s]) for s, r in enumerate(res) if r[0] < INF) and any(r[0] < INF for r in res)
    for o in (st, dec, ref, fst, am):
        o.close()
    ctx.close()


@pytest.mark.gpu
def test_attached_stream_best_path():
    check_attached_stream_best_path()


@pytest.mark.gpu
def test_attached_stream_best_path_eager():
    run_child("import test_gpu_best_path as t\nt.check_attached_stream_best_path()\nprint('CHILD OK')",
              PKB_STREAM_GRAPH="0")


def raw_best_path(ctx, b, fst, n):
    out = [np.zeros(n, np.float64) for _ in range(3)] + [np.zeros(n, np.int32) for _ in range(2)]
    assert ctx.lib.pkb_batch_best_path(b.h, fst.h, 1.0, 1.0, 0.0, *[o.ctypes.data for o in out]) == 0
    return out


@pytest.mark.gpu
def test_arc_overflow_fails_only_its_utterance(ctx):
    am, fst, graph, tid2pdf = make_model(ctx, "loop")
    b, rows = batch_of(ctx, am, LENS)
    n_log = [host_lattice(graph, tid2pdf, r, lattice_beam=4.0)[2] for r in rows]
    big = int(np.argmax(n_log))
    lats, best = b.lattice(fst, lattice_beam=4.0, max_arcs=n_log[big] - 1)
    cost, g, a, nw, nf = raw_best_path(ctx, b, fst, len(rows))
    assert nw[big] == -4 and nf[big] == 0 and math.isnan(cost[big])
    got = b.best_path(fst)
    assert got[big] is None
    check_against_host(got, lats, best, graph, (1.0, 1.0, 0.0), "overflow")
    assert all(len(got[u][5]) == rows[u].shape[0] for u in range(len(rows)) if u != big and got[u][0] < INF)
    for o in (b, fst, am):
        o.close()


@pytest.mark.gpu
def test_epsilon_cycle_fails_each_affected_utterance(ctx):
    am, fst = eps_cycle_model(ctx)
    b, rows = batch_of(ctx, am, [16000, 8000, 0])
    lats, best = b.lattice(fst, lattice_beam=INF)
    cost, g, a, nw, nf = raw_best_path(ctx, b, fst, 3)
    got = b.best_path(fst)
    for u, lat in enumerate(lats):
        assert host_best_path(lat, lattice_T(lat), 0, {}, num_states=fst_states(lat)) == -8, u
        assert nw[u] == -8 and nf[u] == 0 and math.isnan(cost[u]) and got[u] is None
    assert all(x for x in b.nbest(fst, n=4))
    for o in (b, fst, am):
        o.close()


@pytest.mark.gpu
def test_invalid_uses_are_rejected(ctx):
    am, fst, _, _ = make_model(ctx, "loop")
    am2, fst2, _, _ = make_model(ctx, "loop")
    b, _ = batch_of(ctx, am, [16000, 8000])
    with pytest.raises(pk.PkbError):
        b.best_path(fst)                  # no lattice yet
    assert ctx.lib.pkb_batch_best_path_get(b.h, None, None, None) == 1   # before its call
    b.lattice(fst, lattice_beam=4.0)
    assert ctx.lib.pkb_batch_best_path_get(b.h, None, None, None) == 1   # before its call on this lattice
    with pytest.raises(pk.PkbError):
        b.best_path(fst2)                 # another graph
    nan = float("nan")
    for a, g, p in ((0.0, 1.0, 0.0), (-1.0, 1.0, 0.0), (nan, 1.0, 0.0), (INF, 1.0, 0.0), (-INF, 1.0, 0.0),
                    (1.0, -0.5, 0.0), (1.0, nan, 0.0), (1.0, INF, 0.0),
                    (1.0, 1.0, nan), (1.0, 1.0, INF), (1.0, 1.0, -INF)):
        with pytest.raises(pk.PkbError):
            b.best_path(fst, a, g, p)
    outs = [np.zeros(2, np.float64) for _ in range(3)] + [np.zeros(2, np.int32) for _ in range(2)]
    for i in range(5):
        ptrs = [0 if j == i else o.ctypes.data for j, o in enumerate(outs)]
        assert ctx.lib.pkb_batch_best_path(b.h, fst.h, 1.0, 1.0, 0.0, *ptrs) == 1
    assert ctx.lib.pkb_batch_best_path(b.h, fst.h, 1.0, 0.0, -3.0, *[o.ctypes.data for o in outs]) == 0
    assert ctx.lib.pkb_batch_best_path_get(b.h, None, None, None) == 0   # every output may be NULL
    before = bits(b.best_path(fst))
    with pytest.raises(pk.PkbError):
        b.best_path(fst, 0.0)             # refused before it touches the latest results
    assert ctx.lib.pkb_batch_best_path_get(b.h, None, None, None) == 0
    with pytest.raises(pk.PkbError):
        b.lattice(fst, lattice_beam=-1.0)   # refused before it touches the latest lattice
    assert bits(b.best_path(fst)) == before
    b.lattice(fst, lattice_beam=4.0)
    assert ctx.lib.pkb_batch_best_path_get(b.h, None, None, None) == 1   # a new lattice invalidates
    b.close()
    dec = pk.Decoder(ctx, am, fst, 2)
    with pytest.raises(pk.PkbError):
        dec.best_path()                   # before the first finish
    assert ctx.lib.pkb_decoder_best_path_get(dec.h, None, None, None) == 1
    rows = np.zeros((2, 4, am.num_pdfs()), np.float32)
    dec.advance(rows)
    dec.finish()
    with pytest.raises(pk.PkbError):
        dec.best_path()                   # that finish ran without lattices
    dec.set_lattice(4.0)
    dec.advance(rows)
    dec.finish()
    assert ctx.lib.pkb_decoder_best_path_get(dec.h, None, None, None) == 1   # before its call
    assert len(dec.best_path()) == 2
    for a, g, p in ((0.0, 1.0, 0.0), (1.0, -1.0, 0.0), (1.0, 1.0, nan)):
        with pytest.raises(pk.PkbError):
            dec.best_path(a, g, p)
    for i in range(5):
        ptrs = [0 if j == i else o.ctypes.data for j, o in enumerate(outs)]
        assert ctx.lib.pkb_decoder_best_path(dec.h, 1.0, 1.0, 0.0, *ptrs) == 1
    assert ctx.lib.pkb_decoder_best_path_get(dec.h, None, None, None) == 0
    dec.advance(rows)
    with pytest.raises(pk.PkbError):
        dec.best_path()                   # after an advance
    assert ctx.lib.pkb_decoder_best_path_get(dec.h, None, None, None) == 1
    for o in (dec, fst2, am2, fst, am):
        o.close()


@pytest.mark.gpu
def test_best_path_cycles_do_not_leak(ctx):
    import torch
    am, fst, _, _ = make_model(ctx, "loop_big")
    pcm = coloured(7, 16000)

    def cycle():
        b = pk.Batch(ctx, [16000, 16000], synth_global_cmvn(), am, prob_scale=0.1)
        b.set_pcm(np.ascontiguousarray(np.concatenate([pcm, pcm]), np.int16))
        b.run(pk.STAGE_ALL)
        b.lattice(fst, lattice_beam=4.0)
        for tr in TRIPLES:
            res = b.best_path(fst, *tr)
            assert all(np.isfinite(r[0]) and len(r[5]) == b.num_frames[0] for r in res)
        b.close()

    cycle()
    before = torch.cuda.mem_get_info(0)[0]
    for _ in range(20):
        cycle()
    assert before - torch.cuda.mem_get_info(0)[0] <= MARGIN
    fst.close()
    am.close()
