"""N-best lists over lattices (pkb_batch_nbest, pkb_decoder_nbest): the GPU lists must equal, word for
word and bit for bit, a host restatement of the per-node algorithm in the same arithmetic; that
restatement is pinned to brute-force enumeration of lattice paths on tiny graphs."""

import heapq
import math
import os
import sys

import numpy as np
import pytest

import pocketkaldi_b200 as pk
import tools.decode_demo as demo
from oracle.decoder import host_viterbi
from pocketkaldi_b200.synth import synth_global_cmvn

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from test_gpu_lattice import LENS, batch_of, host_lattice, same_records, tiny_graph  # noqa: E402
from test_gpu_online_decode import MARGIN, decode_in_splits, make_model, run_child  # noqa: E402
from test_gpu_online_lattice import stream_rows  # noqa: E402
from test_gpu_viterbi import coloured  # noqa: E402


# ---------------------------------------------------------------- host restatement
def lattice_T(lat):
    emit = lat["t"][lat["ilabel"] != 0]
    return int(emit.max()) + 1 if len(emit) else 0


def host_nbest(lat, T, start, finals, n):
    """The per-node algorithm of csrc/nbest.cu in its arithmetic. A node's list holds up to n entries
    (graph, acoustic, words) with distinct words, ordered by (graph + acoustic, graph, words from the
    last backwards, acoustic). A merge takes inputs (list, w, ac, word), each entry extended to
    (graph + w, acoustic + ac, words + word) in double, and pops the least head over the inputs until
    n distinct word sequences are out. Emitting records of time t merge into the lists of t + 1;
    the epsilon records of a time are Jacobi passes (a destination merges its own list with its
    incoming arcs, all reading the previous pass) until no list changes, at most (records + 1) x
    (n + 1) passes; at T every list, extended by its final weight, merges into the answer. Returns
    [(words, graph, acoustic)] or -6 when a closure did not settle."""
    def merge(inputs):
        heap = []

        def push(i, j):
            lst, w, ac, word = inputs[i]
            if j < len(lst):
                g0, a0, h = lst[j]
                g, a = g0 + w, a0 + ac
                h = h + (word,) if word else h
                heapq.heappush(heap, ((g + a, g, h[::-1], a), i, j, (g, a, h)))

        for i in range(len(inputs)):
            push(i, 0)
        out, seen = [], set()
        while heap and len(out) < n:
            _, i, j, e = heapq.heappop(heap)
            push(i, j + 1)
            if e[2] not in seen:
                seen.add(e[2])
                out.append(e)
        return out

    recs = [(int(r["t"]), int(r["ilabel"]) != 0, int(r["src"]), int(r["dst"]), int(r["olabel"]),
             float(r["graph_cost"]), float(r["acoustic_cost"])) for r in lat]
    groups = {}
    for r in recs:
        groups.setdefault((r[0], r[1]), []).append(r)
    X = {start: [(0.0, 0.0, ())]}
    for t in range(T + 1):
        E = groups.get((t, False), [])
        if E:
            into = {}
            for r in E:
                into.setdefault(r[3], []).append(r)
            max_pass = (len(E) + 1) * (n + 1)
            for p in range(max_pass + 1):
                if p == max_pass:
                    return -6
                new = {d: merge([(X.get(d, []), 0.0, 0.0, 0)] +
                                [(X.get(r[2], []), r[5], r[6], r[4]) for r in rs]) for d, rs in into.items()}
                changed = any(new[d] != X.get(d, []) for d in new)
                X.update(new)
                if not changed:
                    break
        if t == T:
            break
        into = {}
        for r in groups.get((t, True), []):
            into.setdefault(r[3], []).append(r)
        X = {d: merge([(X.get(r[2], []), r[5], r[6], r[4]) for r in rs]) for d, rs in into.items()}
    fin = {s: float(np.float32(v)) for s, v in finals.items()}
    ans = merge([(lst, fin[s], 0.0, 0) for s, lst in X.items() if s in fin])
    return [(list(h), g, a) for g, a, h in ans]


def enumerate_nbest(lat, T, start, finals):
    """Every complete path of the lattice, summed in path order; the best path of each word sequence
    (least cost, then graph); sorted by (cost, graph, words from the last backwards)."""
    out = {}
    for r in lat:
        out.setdefault((int(r["t"]), int(r["src"])), []).append(r)
    best = {}

    def walk(t, s, g, a, words):
        if t == T and s in finals:
            gf = g + float(np.float32(finals[s]))
            k = (gf + a, gf)
            if words not in best or k < best[words][0]:
                best[words] = (k, a)
        for r in out.get((t, s), []):
            w = words + (int(r["olabel"]),) if r["olabel"] else words
            walk(t + (1 if r["ilabel"] else 0), int(r["dst"]), g + float(r["graph_cost"]),
                 a + float(r["acoustic_cost"]), w)

    walk(0, start, 0.0, 0.0, ())
    return sorted(((k[0], k[1], w[::-1], w) for w, (k, _) in best.items()))


def check_against_enumeration(got, want, n):
    assert len(got) == min(n, len(want))
    assert len({tuple(w) for w, _, _ in got}) == len(got)
    for i, (words, g, a) in enumerate(got):
        c = g + a
        assert abs(c - want[i][0]) < 1e-9, (i, got, want[:n])
        # the same sequence, or one whose cost ties with it within 1e-9
        ties = [x for x in want if abs(x[0] - want[i][0]) < 1e-9]
        match = [x for x in ties if list(x[3]) == words]
        assert match, (i, words, ties)
        assert abs(match[0][0] - c) < 1e-9 and abs(match[0][1] - g) < 1e-9


# ---------------------------------------------------------------- CPU: the restatement itself
@pytest.mark.parametrize("seed", range(12))
def test_host_nbest_against_path_enumeration(seed):
    rng = np.random.default_rng(seed)
    graph, tid2pdf = tiny_graph(rng)
    T = int(rng.integers(1, 6))
    loglik = rng.uniform(-3.0, 0.0, (T, 3)).astype(np.float32)
    for lb in (0.5, 2.0, math.inf):
        lat, best, _ = host_lattice(graph, tid2pdf, loglik, beam=1e4, lattice_beam=lb)
        if best == math.inf:
            assert len(lat) == 0
            continue
        want = enumerate_nbest(lat, T, graph[1], graph[2])
        assert want and abs(want[0][0] - best) < 1e-4
        for n in (1, 3, 10, 1000):
            got = host_nbest(lat, lattice_T(lat), graph[1], graph[2], n)
            check_against_enumeration(got, want, n)
        assert len(host_nbest(lat, lattice_T(lat), graph[1], graph[2], 1000)) == len(want)


@pytest.mark.parametrize("seed", range(8))
def test_first_entry_gives_host_viterbi_words(seed):
    rng = np.random.default_rng(100 + seed)
    graph, tid2pdf = demo.word_loop_graph(4, 3, 24) if seed % 2 else tiny_graph(rng, 6)
    P = max(tid2pdf) + 1
    T = int(rng.integers(3, 30))
    loglik = rng.uniform(-6.0, 0.0, (T, P)).astype(np.float32)
    words, _ = host_viterbi(graph, tid2pdf, loglik)
    lat, best, _ = host_lattice(graph, tid2pdf, loglik, lattice_beam=1.0)
    if best == math.inf:
        assert words == []
        return
    got = host_nbest(lat, T, graph[1], graph[2], 3)
    assert got[0][0] == words
    assert abs(got[0][1] + got[0][2] - best) < 1e-3


def test_epsilon_self_loop_with_a_word_converges():
    # (0) -emit-> (1) at t = 0, then an epsilon self-loop on the final state 1 that says word 7
    lat = np.array([(0, 0, 1, 1, 3, 0.25, 1.5), (1, 1, 1, 0, 7, 0.5, 0.0)], pk.LATTICE_ARC_DTYPE)
    got = host_nbest(lat, 1, 0, {1: 0.125}, 4)
    assert [w for w, _, _ in got] == [[3], [3, 7], [3, 7, 7], [3, 7, 7, 7]]
    assert [g for _, g, _ in got] == [0.375, 0.875, 1.375, 1.875]
    assert all(a == 1.5 for _, _, a in got)


# ---------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def ctx():
    c = pk.Context(0)
    yield c
    c.close()


def key(lists):
    """Comparable form of nbest() output, float64 bit patterns included."""
    return [None if x is None else [(w, g.hex(), a.hex()) for w, g, a in x] for x in lists]


def host_lists(lats, best, graph, n):
    return [None if lat is None else [] if best[u] == math.inf else
            host_nbest(lat, lattice_T(lat), graph[1], graph[2], n) for u, lat in enumerate(lats)]


CASES = [(kind, lb, n) for kind in ("loop", "eps") for lb in (0.5, 4.0, math.inf) for n in (1, 4)] + \
        [(kind, 4.0, 64) for kind in ("loop", "eps")] + \
        [(kind, 0.5, n) for kind in ("loop_mid", "loop_big") for n in (1, 4)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,lb,n", CASES)
def test_nbest_equals_the_host_restatement_bitwise(ctx, kind, lb, n):
    am, fst, graph, _ = make_model(ctx, kind)
    lens = LENS + [0] if kind in ("loop", "eps") else [8000, 400, 4000, 0]
    b, rows = batch_of(ctx, am, lens)
    lats, best = b.lattice(fst, lattice_beam=lb)
    got = b.nbest(fst, n=n)
    want = host_lists(lats, best, graph, n)
    assert key(got) == key(want), (kind, lb, n)
    assert n == 1 or any(len(x) > 1 for x in got if x)
    b.close()
    fst.close()
    am.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["loop", "eps", "loop_mid", "loop_big"])
def test_first_entry_is_the_decode_and_calls_change_nothing(ctx, kind):
    am, fst, graph, _ = make_model(ctx, kind)
    b, rows = batch_of(ctx, am, LENS, seed=300)
    hyps, wts = b.decode(fst)
    lats, best = b.lattice(fst, lattice_beam=4.0)
    got = b.nbest(fst, n=4, max_words=3)
    full = b.nbest(fst, n=4)
    assert key(b.nbest(fst, n=4)) == key(full)
    for u in range(len(rows)):
        if not full[u]:
            assert best[u] == math.inf
            continue
        w0, g0, a0 = full[u][0]
        if len(full[u]) < 2 or (full[u][1][1] + full[u][1][2]) - (g0 + a0) > 1e-4:
            assert w0 == hyps[u], (kind, u)
        assert abs(g0 + a0 - best[u]) < 1e-3
        for (w, g, a), (wf, gf, af) in zip(got[u], full[u]):   # truncated to max_words
            assert w == wf[:3] and g == gf and a == af
    lats2, best2 = b.lattice(fst, lattice_beam=4.0)
    assert best2.tobytes() == best.tobytes() and all(same_records(x, y) for x, y in zip(lats, lats2))
    b.nbest(fst, n=4)
    hyps2, wts2 = b.decode(fst)
    assert hyps2 == hyps and wts2.tobytes() == wts.tobytes()
    lats3, _ = b.lattice(fst, lattice_beam=4.0)
    assert all(same_records(x, y) for x, y in zip(lats, lats3))
    b.close()
    fst.close()
    am.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["loop", "eps"])
def test_online_nbest_equals_batch_nbest_for_any_split(ctx, kind):
    am, fst, _, _ = make_model(ctx, kind)
    lens = LENS + [0]
    b, rows = batch_of(ctx, am, lens, seed=500)
    b.lattice(fst, lattice_beam=4.0)
    want = key(b.nbest(fst, n=8))
    b.close()
    T = max(r.shape[0] for r in rows)
    for k in (1, 7, T):
        dec = pk.Decoder(ctx, am, fst, len(lens))
        dec.set_lattice(4.0, max_frames=T)
        with pytest.raises(pk.PkbError):
            dec.nbest()    # no finish yet
        decode_in_splits(dec, rows, k)
        assert key(dec.nbest(n=8)) == want, (kind, k)
        dec.close()
    fst.close()
    am.close()


def check_attached_stream_nbest():
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
        pcm = np.stack([coloured(910 + 10 * rep + s, n) for s in range(S)])
        stream_rows(st, pcm, chunk, rows=False)   # decode-only pushes
        dec.finish()
        got = key(dec.nbest(n=8))
        rows = stream_rows(st, pcm, chunk, rows=True)
        dec.finish()
        ref.advance(np.stack(rows))
        ref.finish()
        assert got == key(ref.nbest(n=8)) == key(dec.nbest(n=8)), rep
        assert all(x for x in got)
    for o in (st, dec, ref, fst, am):
        o.close()
    ctx.close()


@pytest.mark.gpu
def test_attached_stream_nbest():
    check_attached_stream_nbest()


@pytest.mark.gpu
def test_attached_stream_nbest_eager():
    run_child("import test_gpu_nbest as t\nt.check_attached_stream_nbest()\nprint('CHILD OK')",
              PKB_STREAM_GRAPH="0")


@pytest.mark.gpu
def test_arc_overflow_fails_only_its_utterance(ctx):
    am, fst, graph, tid2pdf = make_model(ctx, "loop")
    b, rows = batch_of(ctx, am, LENS)
    host = [host_lattice(graph, tid2pdf, r, lattice_beam=4.0) for r in rows]
    n_log = [h[2] for h in host]
    big = int(np.argmax(n_log))
    lats, best = b.lattice(fst, lattice_beam=4.0, max_arcs=n_log[big] - 1)
    nh = np.zeros(len(rows), np.int32)
    k = len(rows) * 4
    words = np.zeros(k * 16, np.int32)
    nw = np.zeros(k, np.int32)
    g = np.zeros(k, np.float64)
    a = np.zeros(k, np.float64)
    assert ctx.lib.pkb_batch_nbest(b.h, fst.h, 4, 16, words.ctypes.data, nw.ctypes.data, g.ctypes.data,
                                   a.ctypes.data, nh.ctypes.data) == 0
    assert nh[big] == -4
    got = b.nbest(fst, n=4)
    assert key(got) == key(host_lists(lats, best, graph, 4))
    assert got[big] is None and all(got[u] is not None for u in range(len(rows)) if u != big)
    assert any(got[u] for u in range(len(rows)) if u != big)
    b.close()
    fst.close()
    am.close()


@pytest.mark.gpu
def test_invalid_uses_are_rejected(ctx):
    am, fst, graph, _ = make_model(ctx, "loop")
    am2, fst2, _, _ = make_model(ctx, "loop")
    b, _ = batch_of(ctx, am, [16000, 8000])
    with pytest.raises(pk.PkbError):
        b.nbest(fst)                 # no lattice yet
    b.lattice(fst, lattice_beam=4.0)
    for n, mw in ((0, 8), (1025, 8), (-1, 8), (4, 0), (4, -2)):
        with pytest.raises(pk.PkbError):
            b.nbest(fst, n=n, max_words=mw)
    with pytest.raises(pk.PkbError):
        b.nbest(fst2)                # another graph
    outs = [np.zeros(2 * 4 * 8, np.int32), np.zeros(8, np.int32), np.zeros(8), np.zeros(8), np.zeros(2, np.int32)]
    for i in range(5):
        ptrs = [0 if j == i else o.ctypes.data for j, o in enumerate(outs)]
        assert ctx.lib.pkb_batch_nbest(b.h, fst.h, 4, 8, *ptrs) == 1  # PKB_ERR_INVALID
        assert ctx.lib.pkb_batch_nbest(b.h, fst.h, 4, 8, *[o.ctypes.data for o in outs]) == 0
    assert b.nbest(fst, n=1024) is not None and b.nbest(fst, n=1, max_words=1) is not None
    before = key(b.nbest(fst))
    with pytest.raises(pk.PkbError):
        b.lattice(fst, lattice_beam=-1.0)   # refused before it touches the latest lattice
    assert key(b.nbest(fst)) == before
    b.close()
    dec = pk.Decoder(ctx, am, fst, 2)
    rows = np.zeros((2, 4, am.num_pdfs()), np.float32)
    dec.advance(rows)
    dec.finish()
    with pytest.raises(pk.PkbError):
        dec.nbest()                  # that finish ran without lattices
    dec.set_lattice(4.0)
    dec.advance(rows)
    dec.finish()
    assert len(dec.nbest(n=2)) == 2
    for n, mw in ((0, 8), (1025, 8), (4, 0)):
        with pytest.raises(pk.PkbError):
            dec.nbest(n=n, max_words=mw)
    for i in range(5):
        ptrs = [0 if j == i else o.ctypes.data for j, o in enumerate(outs)]
        assert ctx.lib.pkb_decoder_nbest(dec.h, 4, 8, *ptrs) == 1  # PKB_ERR_INVALID
    dec.advance(rows)
    with pytest.raises(pk.PkbError):
        dec.nbest()                  # after an advance
    dec.close()
    fst2.close()
    am2.close()
    fst.close()
    am.close()


@pytest.mark.gpu
def test_nbest_cycles_do_not_leak(ctx):
    import torch
    am, fst, _, _ = make_model(ctx, "loop_big")
    pcm = coloured(7, 16000)

    def cycle():
        b = pk.Batch(ctx, [16000, 16000], synth_global_cmvn(), am, prob_scale=0.1)
        b.set_pcm(np.ascontiguousarray(np.concatenate([pcm, pcm]), np.int16))
        b.run(pk.STAGE_ALL)
        b.lattice(fst, lattice_beam=4.0)
        got = b.nbest(fst, n=16)
        assert all(x for x in got)
        b.close()

    cycle()
    before = torch.cuda.mem_get_info(0)[0]
    for _ in range(20):
        cycle()
    assert before - torch.cuda.mem_get_info(0)[0] <= MARGIN
    fst.close()
    am.close()
