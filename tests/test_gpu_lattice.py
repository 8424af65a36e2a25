"""Lattices of the batch search (pkb_batch_lattice): the arcs the GPU keeps must equal, record for
record and bit for bit, a host restatement of the lattice in the search's own arithmetic; that
restatement is pinned to brute-force path enumeration on tiny graphs. The best path through a
lattice gives the words of pkb_batch_decode, and overflow is reported per utterance."""

import math
import os
import shutil
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

LENS = [16000, 24000, 8000, 32000, 400, 12345]
MARGIN = 64 << 20


# ---------------------------------------------------------------- host restatement
def host_lattice(graph, tid2pdf, loglik, beam=16.0, lattice_beam=8.0):
    """The lattice of the GPU search in its arithmetic (oracle/decoder.host_viterbi's, with arcs
    indexed in the sorted order pk.Fst gives them): nodes (t, s) carry the float token costs alpha;
    an emitting arc is included when alpha(t, src) <= float(best + beam) and its double total is
    within the next cutoff, an epsilon arc when alpha(t, src) + w is within the closure bound of t.
    beta(T, s) = final(s), beta(t, s) = min over included arcs leaving (t, s) of (w + ac) +
    beta(head), epsilon arcs of a time relaxed to a fixpoint; an arc is kept when beta(head) is
    finite and ((alpha(tail) + w) + ac) + beta(head) <= best + lattice_beam. Returns (records in
    output order as LATTICE_ARC_DTYPE, best, number of included arcs)."""
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
        wc = float(np.float32(alpha[np.isfinite(alpha)].min() + beam))
        ac = -np.asarray(row, np.float32)[pdf].astype(np.float64)
        tot = (alpha[src] + w) + ac
        m = emit & (alpha[src] <= wc)
        if not m.any():
            return empty, math.inf, sum(len(g) for g in g_eps + g_emit)
        nc = tot[m].min() + beam
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


def lattice_best_path(lat, T, start, finals):
    """The search's 1-best over the arcs of a lattice: float costs, a token replaced only by a
    strictly lower cost, emitting arcs in arc order before the epsilon closure of the next time.
    Returns (words, end state, float cost of the end token), or None without a final token."""
    f32 = lambda x: float(np.float32(x))
    cur = {start: (0.0, ())}
    for t in range(T + 1):
        here = lat[lat["t"] == t]
        eps = here[here["ilabel"] == 0]
        changed = True
        while changed:
            changed = False
            for r in eps:
                if int(r["src"]) not in cur:
                    continue
                c0, words = cur[int(r["src"])]
                c = f32(c0 + float(r["graph_cost"]))
                d = int(r["dst"])
                if d not in cur or c < cur[d][0]:
                    cur[d] = (c, words + (int(r["olabel"]),) if r["olabel"] else words)
                    changed = True
        if t == T:
            break
        new = {}
        for r in here[here["ilabel"] != 0]:
            if int(r["src"]) not in cur:
                continue
            c0, words = cur[int(r["src"])]
            c = f32((c0 + float(r["graph_cost"])) + float(r["acoustic_cost"]))
            d = int(r["dst"])
            if d not in new or c < new[d][0]:
                new[d] = (c, words + (int(r["olabel"]),) if r["olabel"] else words)
        cur = new
    ends = [(f32(c + finals[s]), s, c, words) for s, (c, words) in cur.items() if s in finals]
    if not ends:
        return None
    _, s, c, words = min(ends)
    return list(words), s, c


# ---------------------------------------------------------------- CPU: the restatement itself
def tiny_graph(rng, n_states=5):
    """Random acyclic-in-epsilon graph: emitting arcs anywhere, epsilon arcs to higher states."""
    arcs = []
    for s in range(n_states):
        for _ in range(rng.integers(1, 4)):
            arcs.append((s, int(rng.integers(0, n_states)), int(rng.integers(1, 4)), int(rng.integers(0, 3)),
                         float(np.float32(rng.uniform(0.0, 1.0)))))
        if s + 1 < n_states and rng.random() < 0.5:
            arcs.append((s, int(rng.integers(s + 1, n_states)), 0, int(rng.integers(0, 3)),
                         float(np.float32(rng.uniform(0.0, 1.0)))))
    finals = {s: float(np.float32(rng.uniform(0.0, 0.5))) for s in range(n_states) if rng.random() < 0.5}
    finals.setdefault(n_states - 1, 0.25)
    return (n_states, 0, finals, arcs), [0, 0, 1, 2]


def brute_force(graph, tid2pdf, loglik):
    """Best complete path cost through every arc occurrence (t, arc index), by enumeration."""
    num_states, start, finals, arcs = graph
    arcs = sorted(arcs)
    out = [[] for _ in range(num_states)]
    for i, (s, d, i_l, o_l, wt) in enumerate(arcs):
        out[s].append((i, d, i_l, float(np.float32(wt))))
    T = len(loglik)
    through, best = {}, [math.inf]

    def walk(t, s, cost, used):
        if t == T and s in finals:
            c = cost + float(np.float32(finals[s]))
            best[0] = min(best[0], c)
            for key in used:
                through[key] = min(through.get(key, math.inf), c)
        for i, d, i_l, wt in out[s]:
            if i_l == 0:
                walk(t, d, cost + wt, used + ((t, i),))
            elif t < T:
                walk(t + 1, d, cost + wt - float(loglik[t][tid2pdf[i_l]]), used + ((t, i),))

    walk(0, start, 0.0, ())
    return through, best[0]


@pytest.mark.parametrize("seed", range(12))
def test_host_lattice_against_path_enumeration(seed):
    rng = np.random.default_rng(seed)
    graph, tid2pdf = tiny_graph(rng)
    T = int(rng.integers(1, 6))
    loglik = rng.uniform(-3.0, 0.0, (T, 3)).astype(np.float32)
    through, best = brute_force(graph, tid2pdf, loglik)
    arcs = sorted(graph[3])
    index = {(a[0], a[1], a[2], a[3], float(np.float32(a[4]))): i for i, a in enumerate(arcs)}
    for lb in (0.5, 2.0, math.inf):
        lat, hbest, _ = host_lattice(graph, tid2pdf, loglik, beam=1e4, lattice_beam=lb)
        if best == math.inf:
            assert hbest == math.inf and len(lat) == 0
            continue
        assert abs(hbest - best) < 1e-4
        kept = {(int(r["t"]), index[(int(r["src"]), int(r["dst"]), int(r["ilabel"]), int(r["olabel"]),
                                     float(r["graph_cost"]))]) for r in lat}
        assert len(kept) == len(lat)
        for key, c in through.items():
            if c <= best + lb - 1e-4:
                assert key in kept, (seed, lb, key, c, best)
            elif c >= best + lb + 1e-4:
                assert key not in kept, (seed, lb, key, c, best)
        assert kept <= set(through)  # every kept arc lies on a complete path
        # output order: by time, epsilon arcs first, then arc index
        keys = [(int(r["t"]), int(r["ilabel"]) != 0,
                 index[(int(r["src"]), int(r["dst"]), int(r["ilabel"]), int(r["olabel"]), float(r["graph_cost"]))])
                for r in lat]
        assert keys == sorted(keys)


@pytest.mark.parametrize("seed", range(8))
def test_best_path_through_the_host_lattice_gives_host_viterbi_words(seed):
    rng = np.random.default_rng(100 + seed)
    graph, tid2pdf = demo.word_loop_graph(4, 3, 24) if seed % 2 else tiny_graph(rng, 6)
    P = max(tid2pdf) + 1
    T = int(rng.integers(3, 30))
    loglik = rng.uniform(-6.0, 0.0, (T, P)).astype(np.float32)
    words, weight = host_viterbi(graph, tid2pdf, loglik)
    lat, best, _ = host_lattice(graph, tid2pdf, loglik, lattice_beam=1.0)
    bp = lattice_best_path(lat, T, graph[1], graph[2])
    if best == math.inf:
        assert bp is None and words == [] and weight == 0.0
        return
    got, s, c = bp
    assert got == words
    assert np.float32(np.float32(best) + np.float32(graph[2][s])) == np.float32(weight)


def test_lattice_arc_record_is_28_bytes():
    assert pk.LATTICE_ARC_DTYPE.itemsize == 28
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        c_file = os.path.join(d, "size.c")
        with open(c_file, "w") as f:
            f.write('#include <stddef.h>\n#include <stdio.h>\n#include "pkb200.h"\n'
                    'int main(void) { printf("%zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(pkb_lattice_arc_t), '
                    'offsetof(pkb_lattice_arc_t, t), offsetof(pkb_lattice_arc_t, src), '
                    'offsetof(pkb_lattice_arc_t, dst), offsetof(pkb_lattice_arc_t, ilabel), '
                    'offsetof(pkb_lattice_arc_t, olabel), offsetof(pkb_lattice_arc_t, graph_cost), '
                    'offsetof(pkb_lattice_arc_t, acoustic_cost)); return 0; }\n')
        exe = os.path.join(d, "size")
        subprocess.check_call([cc, "-std=c99", "-I", os.path.join(ROOT, "include"), "-o", exe, c_file])
        got = [int(x) for x in subprocess.check_output([exe]).split()]
    dt = pk.LATTICE_ARC_DTYPE
    assert got == [dt.itemsize] + [dt.fields[n][1] for n in dt.names]


# ---------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def ctx():
    c = pk.Context(0)
    yield c
    c.close()


def coloured(seed, n):
    from test_gpu_viterbi import coloured as col
    return col(seed, n)


def make_model(ctx, kind):
    from test_gpu_online_decode import make_model as mm
    return mm(ctx, kind)


def batch_of(ctx, am, lens, seed=100):
    pcms = [coloured(seed + u, n) if n else np.zeros(0, np.int16) for u, n in enumerate(lens)]
    b = pk.Batch(ctx, lens, synth_global_cmvn(), am, prob_scale=0.1)
    if sum(lens):
        b.set_pcm(np.ascontiguousarray(np.concatenate(pcms), np.int16))
    b.run(pk.STAGE_ALL)
    ll = b.get(pk.BUF_LOGLIK)
    off = np.concatenate([[0], np.cumsum(b.num_frames)])
    rows = [ll[off[u]:off[u + 1]].copy() for u in range(len(lens))]
    return b, rows


def same_records(a, b):
    return a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["loop", "eps", "loop_mid", "loop_big"])
def test_lattice_equals_the_host_restatement_bitwise(ctx, kind):
    am, fst, graph, tid2pdf = make_model(ctx, kind)
    b, rows = batch_of(ctx, am, LENS + [0])
    for lb in (0.5, 4.0, math.inf):
        lats, best = b.lattice(fst, lattice_beam=lb)
        for u, r in enumerate(rows):
            want, wbest, _ = host_lattice(graph, tid2pdf, r, lattice_beam=lb)
            assert lats[u] is not None, (kind, lb, u)
            assert same_records(lats[u], want), (kind, lb, u, len(lats[u]), len(want))
            assert np.float64(best[u]).tobytes() == np.float64(wbest).tobytes(), (kind, lb, u, best[u], wbest)
        assert any(len(x) > 0 for x in lats)
    b.close()
    fst.close()
    am.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["loop", "eps", "loop_mid", "loop_big"])
def test_lattice_best_path_and_decode_agree(ctx, kind):
    am, fst, graph, _ = make_model(ctx, kind)
    b, rows = batch_of(ctx, am, LENS, seed=300)
    hyps, wts = b.decode(fst)
    lats, best = b.lattice(fst, lattice_beam=4.0)
    lats2, best2 = b.lattice(fst, lattice_beam=4.0)
    hyps2, wts2 = b.decode(fst)
    assert hyps2 == hyps and wts2.tobytes() == wts.tobytes()
    assert best2.tobytes() == best.tobytes()
    assert all(same_records(x, y) for x, y in zip(lats, lats2))
    finals = graph[2]
    for u, r in enumerate(rows):
        bp = lattice_best_path(lats[u], r.shape[0], graph[1], finals)
        if bp is None:
            assert hyps[u] == [] and best[u] == math.inf
            continue
        words, s, c = bp
        assert words == hyps[u], (kind, u)
        assert best[u] == float(np.float32(c)) + float(np.float32(finals[s]))
        # BestPath adds the final weight twice, in float
        assert np.float32(np.float32(best[u]) + np.float32(finals[s])) == wts[u]
    b.close()
    fst.close()
    am.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["loop", "loop_big"])
def test_arc_overflow_fails_only_its_utterance(ctx, kind):
    am, fst, graph, tid2pdf = make_model(ctx, kind)
    b, rows = batch_of(ctx, am, LENS)
    host = [host_lattice(graph, tid2pdf, r, lattice_beam=4.0) for r in rows]
    n_log = [h[2] for h in host]
    big = int(np.argmax(n_log))
    assert sorted(n_log)[-2] < n_log[big]
    lats, best = b.lattice(fst, lattice_beam=4.0, max_arcs=n_log[big] - 1)
    for u in range(len(rows)):
        if u == big:
            assert lats[u] is None and best[u] == math.inf
        else:
            assert same_records(lats[u], host[u][0])
    lib = ctx.lib
    na = np.zeros(len(rows), np.int64)
    bc = np.zeros(len(rows), np.float64)
    assert lib.pkb_batch_lattice(b.h, fst.h, 0.0, 4.0, 0, n_log[big] - 1, na.ctypes.data, bc.ctypes.data) == 0
    assert na[big] == -4
    lats, _ = b.lattice(fst, lattice_beam=4.0, max_arcs=n_log[big])  # the next call is clean
    assert all(same_records(lats[u], host[u][0]) for u in range(len(rows)))
    b.close()
    fst.close()
    am.close()


@pytest.mark.gpu
def test_token_overflow_is_reported_and_the_next_call_is_exact(ctx):
    rng = np.random.default_rng(3)
    P = 640
    layers = formats.make_dnn(rng, 440, 32, 1, P)
    prior = np.full(P, 1.0 / P, np.float32)
    graph, tid2pdf = demo.word_loop_graph(200, 3, P)   # 601 states: tables in the global workspace
    am = pk.AcousticModel(ctx, pk.PREC_BF16X3).from_layers(layers, prior, 5, 5, tid2pdf=tid2pdf)
    fst = pk.Fst(ctx, graph=graph)
    from pocketkaldi_b200.synth import synth_pcm
    pcms = [synth_pcm(5, [0], 16000)[0], synth_pcm(5, [1], 16000)[0]]
    b = pk.Batch(ctx, [16000, 16000], synth_global_cmvn(), am, prob_scale=0.1)
    b.set_pcm(np.ascontiguousarray(np.concatenate(pcms), np.int16))
    b.run(pk.STAGE_ALL)
    na = np.zeros(2, np.int64)
    bc = np.zeros(2, np.float64)
    assert ctx.lib.pkb_batch_lattice(b.h, fst.h, 0.0, 4.0, 64, 0, na.ctypes.data, bc.ctypes.data) == 0
    assert list(na) == [-1, -1]
    lats, best = b.lattice(fst, lattice_beam=4.0, max_tokens=1024)
    ll = b.get(pk.BUF_LOGLIK)
    rows = [ll[:b.num_frames[0]], ll[b.num_frames[0]:]]
    for u in range(2):
        want, wbest, _ = host_lattice(graph, tid2pdf, rows[u], lattice_beam=4.0)
        assert same_records(lats[u], want) and best[u] == wbest
    b.close()
    fst.close()
    am.close()


@pytest.mark.gpu
def test_invalid_uses_are_rejected(ctx):
    am, fst, graph, tid2pdf = make_model(ctx, "loop")
    b, _ = batch_of(ctx, am, [16000])
    for lb in (0.0, -1.0, float("nan")):
        with pytest.raises(pk.PkbError):
            b.lattice(fst, lattice_beam=lb)
    b.set_compact(True)
    with pytest.raises(pk.PkbError):
        b.lattice(fst)
    with pytest.raises(pk.PkbError):
        b.decode(fst)
    b.close()
    rng = np.random.default_rng(1)
    layers = formats.make_dnn(rng, 440, 96, 2, 96)
    bare = pk.AcousticModel(ctx, pk.PREC_BF16X3).from_layers(layers, np.full(96, 1.0 / 96, np.float32), 5, 5)
    b2, _ = batch_of(ctx, bare, [16000])
    with pytest.raises(pk.PkbError):
        b2.lattice(fst)
    b2.close()
    bare.close()
    fst.close()
    am.close()


@pytest.mark.gpu
def test_batches_with_lattices_do_not_leak(ctx):
    import torch
    am, fst, _, _ = make_model(ctx, "loop_big")
    pcm = coloured(7, 16000)

    def cycle():
        b = pk.Batch(ctx, [16000, 16000], synth_global_cmvn(), am, prob_scale=0.1)
        b.set_pcm(np.ascontiguousarray(np.concatenate([pcm, pcm]), np.int16))
        b.run(pk.STAGE_ALL)
        lats, _ = b.lattice(fst, lattice_beam=4.0)
        assert all(x is not None and len(x) for x in lats)
        b.close()

    cycle()
    before = torch.cuda.mem_get_info(0)[0]
    for _ in range(20):
        cycle()
    assert before - torch.cuda.mem_get_info(0)[0] <= MARGIN
    fst.close()
    am.close()
