"""Arc and frame posteriors over lattices (pkb_batch_posteriors, pkb_decoder_posteriors): the GPU
results must match a host restatement of the forward-backward pass in the fold order of
include/pkb200.h; that restatement is pinned to brute-force enumeration of lattice paths, and of
graph paths, on tiny graphs."""

import math
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

import pocketkaldi_b200 as pk
from pocketkaldi_b200 import formats
from pocketkaldi_b200.synth import synth_global_cmvn

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
from test_gpu_lattice import LENS, batch_of, brute_force, host_lattice, same_records, tiny_graph  # noqa: E402
from test_gpu_nbest import key as nbest_key, lattice_T  # noqa: E402
from test_gpu_online_decode import MARGIN, decode_in_splits, make_model, run_child  # noqa: E402
from test_gpu_online_lattice import stream_rows  # noqa: E402
from test_gpu_viterbi import coloured, eps_graph  # noqa: E402

INF = math.inf


# ---------------------------------------------------------------- host restatement
def lse(a, b):
    """-log(exp(-a) + exp(-b)) elementwise, +inf the identity."""
    m, M = np.minimum(a, b), np.maximum(a, b)
    with np.errstate(invalid="ignore", over="ignore"):
        return np.where(M == INF, m, m - np.log1p(np.exp(m - M)))


def fold(acc, node, val, op=lse):
    """acc[node[i]] = op(acc[node[i]], val[i]) for every i, each node's values in ascending i."""
    acc = acc.copy()
    if len(node) == 0:
        return acc
    order = np.argsort(node, kind="stable")
    n_sorted = node[order]
    start = np.r_[0, np.nonzero(np.diff(n_sorted))[0] + 1]
    rank = np.arange(len(order)) - np.repeat(start, np.diff(np.r_[start, len(order)]))
    by_rank = order[np.argsort(rank, kind="stable")]
    bounds = np.r_[0, np.cumsum(np.bincount(rank))]
    for j in range(len(bounds) - 1):
        sel = by_rank[bounds[j]:bounds[j + 1]]
        acc[node[sel]] = op(acc[node[sel]], val[sel])
    return acc


def host_posteriors(lat, T, start, finals, tid2pdf, acoustic_scale=1.0, graph_scale=1.0, min_post=0.0,
                    num_states=None):
    """The forward-backward pass of include/pkb200.h in its fold order: alpha folds a node's
    incoming records in record order, beta its outgoing records (epsilon, then emitting) in record
    order, the epsilon records of a time in Kahn levels. Returns (total, arc posteriors as float64,
    [(t, pdf, float32 post)] in (t, pdf) order), or (-8, None, None) for an epsilon cycle."""
    S = num_states or (max([start] + list(finals) + [int(x) for x in lat["src"]] +
                           [int(x) for x in lat["dst"]]) + 1)
    as_, gs = float(np.float32(acoustic_scale)), float(np.float32(graph_scale))
    t_, src, dst = lat["t"].astype(np.int64), lat["src"].astype(np.int64), lat["dst"].astype(np.int64)
    emit = lat["ilabel"] != 0
    c = gs * lat["graph_cost"].astype(np.float64) + as_ * lat["acoustic_cost"].astype(np.float64)
    fin = np.full(S, INF)
    for s, v in finals.items():
        fin[s] = gs * float(np.float32(v))
    pdf = np.asarray(tid2pdf, np.int64)[lat["ilabel"]]
    # records come sorted by group 2 t + emitting
    bounds = np.searchsorted(2 * t_ + emit, np.arange(2 * T + 3))
    groups = {(t, e): np.arange(bounds[2 * t + e], bounds[2 * t + e + 1]) for t in range(T + 1) for e in (0, 1)}

    alpha_rec = np.full(len(lat), INF)
    X = np.full(S, INF)
    X[start] = 0.0
    for t in range(T + 1):
        E = groups[(t, 0)]
        done = np.ones(S, bool)
        done[dst[E]] = False
        while not done.all():
            inc_ok = np.ones(S, bool)
            np.logical_and.at(inc_ok, dst[E], done[src[E]])
            ready = ~done & inc_ok
            if not ready.any():
                return -8, None, None
            r = E[ready[dst[E]]]
            X = fold(X, dst[r], X[src[r]] + c[r])
            done |= ready
        M = groups[(t, 1)] if t < T else np.zeros(0, np.int64)
        for g in (E, M):
            alpha_rec[g] = X[src[g]]
        if t == T:
            break
        X = fold(np.full(S, INF), dst[M], X[src[M]] + c[M])
    total = INF
    for s in sorted(finals):
        total = float(lse(total, X[s] + fin[s]))

    post = np.zeros(len(lat))
    frames = []
    Bn = None
    for t in range(T, -1, -1):
        E = groups[(t, 0)]
        M = groups[(t, 1)] if t < T else np.zeros(0, np.int64)
        if len(M):
            with np.errstate(over="ignore"):
                post[M] = np.exp(total - ((alpha_rec[M] + c[M]) + Bn[dst[M]])) if total < INF else 0.0
            sums = fold(np.zeros(int(pdf.max()) + 1), pdf[M], post[M], op=np.add)
            frames_t = [(t, int(p), np.float32(sums[p])) for p in sorted(set(pdf[M].tolist()))]
            frames = [f for f in frames_t if f[2] >= np.float32(min_post)] + frames
        base = fin.copy() if t == T else np.full(S, INF)
        B = np.full(S, INF)
        done = np.zeros(S, bool)
        while not done.all():
            out_ok = np.ones(S, bool)
            np.logical_and.at(out_ok, src[E], done[dst[E]])
            ready = ~done & out_ok
            assert ready.any()
            b = base.copy()
            re_ = E[ready[src[E]]]
            b = fold(b, src[re_], c[re_] + B[dst[re_]])
            if len(M):
                rm = M[ready[src[M]]]
                b = fold(b, src[rm], c[rm] + Bn[dst[rm]])
            B[ready] = b[ready]
            done |= ready
        if len(E):
            with np.errstate(over="ignore"):
                post[E] = np.exp(total - ((alpha_rec[E] + c[E]) + B[dst[E]])) if total < INF else 0.0
        Bn = B
    return total, post, frames


def enumerate_posteriors(lat, T, start, finals, acoustic_scale, graph_scale):
    """Every complete path of the lattice: -log of the sum of exp(-cost), and per record the share
    of that sum through it."""
    as_, gs = float(np.float32(acoustic_scale)), float(np.float32(graph_scale))
    out = {}
    for i, r in enumerate(lat):
        out.setdefault((int(r["t"]), int(r["src"])), []).append(i)
    paths = []

    def walk(t, s, cost, used):
        if t == T and s in finals:
            paths.append((cost + gs * float(np.float32(finals[s])), used))
        for i in out.get((t, s), []):
            r = lat[i]
            c = gs * float(r["graph_cost"]) + as_ * float(r["acoustic_cost"])
            walk(t + (1 if r["ilabel"] else 0), int(r["dst"]), cost + c, used + (i,))

    walk(0, start, 0.0, ())
    if not paths:
        return INF, np.zeros(len(lat))
    lo = min(p[0] for p in paths)
    w = [math.exp(lo - p[0]) for p in paths]
    total = lo - math.log(math.fsum(w))
    post = np.zeros(len(lat))
    for (cost, used), _ in zip(paths, w):
        for i in used:
            post[i] += math.exp(total - cost)
    return total, post


def graph_total(graph, tid2pdf, loglik, acoustic_scale, graph_scale):
    """-log of the sum over every complete path of the graph (no pruning)."""
    num_states, start, finals, arcs = graph
    as_, gs = float(np.float32(acoustic_scale)), float(np.float32(graph_scale))
    T = len(loglik)
    costs = []

    def walk(t, s, cost):
        if t == T and s in finals:
            costs.append(cost + gs * float(np.float32(finals[s])))
        for (a, d, il, ol, w) in arcs:
            if a != s:
                continue
            if il == 0:
                walk(t, d, cost + gs * float(np.float32(w)))
            elif t < T:
                ac = float(np.float32(-np.float32(loglik[t][tid2pdf[il]])))
                walk(t + 1, d, cost + (gs * float(np.float32(w)) + as_ * ac))

    walk(0, start, 0.0)
    lo = min(costs)
    return lo - math.log(math.fsum(math.exp(lo - c) for c in costs))


def close(a, b, rel):
    return a == b or abs(a - b) <= rel * max(abs(a), abs(b))


# ---------------------------------------------------------------- CPU: the restatement itself
@pytest.mark.parametrize("seed", range(12))
def test_host_posteriors_against_path_enumeration(seed):
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
        for scales in ((1.0, 1.0), (0.3, 1.5)):
            total, post, frames = host_posteriors(lat, lattice_T(lat), graph[1], graph[2], tid2pdf, *scales,
                                                  num_states=graph[0])
            want_total, want_post = enumerate_posteriors(lat, lattice_T(lat), graph[1], graph[2], *scales)
            assert close(total, want_total, 1e-12), (seed, lb, scales, total, want_total)
            for i in range(len(lat)):
                assert close(post[i], want_post[i], 1e-12), (seed, lb, scales, i, post[i], want_post[i])
            if lb == INF:
                assert lattice_T(lat) == T
                assert close(total, graph_total(graph, tid2pdf, loglik, *scales), 1e-12), (seed, scales)


@pytest.mark.parametrize("seed", range(8))
def test_posteriors_of_each_frame_sum_to_one(seed):
    rng = np.random.default_rng(50 + seed)
    graph, tid2pdf = tiny_graph(rng, 6)
    T = int(rng.integers(2, 8))
    loglik = rng.uniform(-3.0, 0.0, (T, 3)).astype(np.float32)
    lat, best, _ = host_lattice(graph, tid2pdf, loglik, beam=1e4, lattice_beam=INF)
    if best == INF:
        return
    total, post, frames = host_posteriors(lat, T, graph[1], graph[2], tid2pdf, 0.3, 1.5, num_states=graph[0])
    emit = lat["ilabel"] != 0
    for t in range(T):
        m = emit & (lat["t"] == t)
        assert abs(math.fsum(post[m]) - 1.0) < 1e-12, (seed, t)
        assert abs(math.fsum(float(p) for tt, _, p in frames if tt == t) - 1.0) < 1e-6
    assert [(t, p) for t, p, _ in frames] == sorted((t, p) for t, p, _ in frames)
    for mp in (1e-3, 0.2, 0.5, 1.0):
        _, _, kept = host_posteriors(lat, T, graph[1], graph[2], tid2pdf, 0.3, 1.5, mp, num_states=graph[0])
        assert kept == [f for f in frames if f[2] >= np.float32(mp)]


def test_epsilon_cycles_give_minus_8():
    # the epsilon self-loop of test_gpu_nbest.py, and a two-state cycle
    loop = np.array([(0, 0, 1, 1, 3, 0.25, 1.5), (1, 1, 1, 0, 7, 0.5, 0.0)], pk.LATTICE_ARC_DTYPE)
    assert host_posteriors(loop, 1, 0, {1: 0.125}, [0, 0])[0] == -8
    two = np.array([(0, 0, 1, 1, 3, 0.25, 1.5), (1, 1, 2, 0, 0, 0.5, 0.0), (1, 2, 1, 0, 0, 0.5, 0.0)],
                   pk.LATTICE_ARC_DTYPE)
    assert host_posteriors(two, 1, 0, {1: 0.125}, [0, 0])[0] == -8
    chain = two[:2]   # without the way back: a plain lattice
    total, post, frames = host_posteriors(chain, 1, 0, {1: 0.125, 2: 0.0}, [0, 0])
    assert np.allclose(post, [1.0, float(np.exp(-0.5) / (np.exp(-0.125) + np.exp(-0.5)))], rtol=1e-12)


def test_frame_post_record_is_12_bytes():
    assert pk.FRAME_POST_DTYPE.itemsize == 12
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        c_file = os.path.join(d, "size.c")
        with open(c_file, "w") as f:
            f.write('#include <stddef.h>\n#include <stdio.h>\n#include "pkb200.h"\n'
                    'int main(void) { printf("%zu %zu %zu %zu\\n", sizeof(pkb_frame_post_t), '
                    'offsetof(pkb_frame_post_t, t), offsetof(pkb_frame_post_t, pdf), '
                    'offsetof(pkb_frame_post_t, post)); return 0; }\n')
        exe = os.path.join(d, "size")
        subprocess.check_call([cc, "-std=c99", "-I", os.path.join(ROOT, "include"), "-o", exe, c_file])
        got = [int(x) for x in subprocess.check_output([exe]).split()]
    dt = pk.FRAME_POST_DTYPE
    assert got == [dt.itemsize] + [dt.fields[n][1] for n in dt.names]


# ---------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def ctx():
    c = pk.Context(0)
    yield c
    c.close()


def bits(res):
    """Comparable form of posteriors() output, bit patterns included."""
    tot, arcs, frames = res
    return (tot.tobytes(), [None if a is None else a.tobytes() for a in arcs],
            [None if f is None else f.tobytes() for f in frames])


def check_against_host(got, lats, best, graph, tid2pdf, scales, min_post, where):
    tot, arcs, frames = got
    for u, lat in enumerate(lats):
        if lat is None:
            assert arcs[u] is None and frames[u] is None
            continue
        if best[u] == INF:
            assert tot[u] == INF and len(arcs[u]) == 0 and len(frames[u]) == 0
            continue
        T = lattice_T(lat)
        w_tot, w_post, w_frames = host_posteriors(lat, T, graph[1], graph[2], tid2pdf, *scales, 0.0,
                                                  num_states=graph[0])
        assert abs(tot[u] - w_tot) <= 1e-9 * max(1.0, abs(w_tot)), (where, u, tot[u], w_tot)
        assert len(arcs[u]) == len(lat)
        assert np.abs(arcs[u].astype(np.float64) - w_post).max(initial=0.0) <= 1e-6, (where, u)
        g = {(int(f["t"]), int(f["pdf"])): float(f["post"]) for f in frames[u]}
        assert [(int(f["t"]), int(f["pdf"])) for f in frames[u]] == sorted(g)
        for t, p, v in w_frames:
            v = float(v)
            if abs(v - min_post) <= 1e-6:
                continue
            if v >= min_post:
                assert (t, p) in g and abs(g[(t, p)] - v) <= 1e-6, (where, u, t, p, v, g.get((t, p)))
            else:
                assert (t, p) not in g, (where, u, t, p, v)
        assert all(v >= np.float32(min_post) for v in g.values())
        for t in range(T):
            m = (lat["t"] == t) & (lat["ilabel"] != 0)
            assert abs(float(arcs[u][m].astype(np.float64).sum()) - 1.0) < 1e-4, (where, u, t)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["loop", "eps", "loop_mid", "loop_big"])
@pytest.mark.parametrize("lb", [0.5, 4.0, INF])
def test_posteriors_match_the_host_restatement(ctx, kind, lb):
    am, fst, graph, tid2pdf = make_model(ctx, kind)
    b, rows = batch_of(ctx, am, LENS + [0])
    lats, best = b.lattice(fst, lattice_beam=lb)
    for scales in ((1.0, 1.0), (0.3, 1.5)):
        for min_post in (0.0, 1e-3):
            got = b.posteriors(fst, *scales, min_post=min_post)
            check_against_host(got, lats, best, graph, tid2pdf, scales, min_post, (kind, lb, scales, min_post))
    assert len(lats[-1]) == 0 or lattice_T(lats[-1]) == 0
    b.close()
    fst.close()
    am.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["loop", "eps", "loop_big"])
def test_repeated_calls_are_identical_and_change_nothing(ctx, kind):
    am, fst, _, _ = make_model(ctx, kind)
    b, rows = batch_of(ctx, am, LENS, seed=300)
    hyps, wts = b.decode(fst)
    lats, best = b.lattice(fst, lattice_beam=4.0)
    nb = nbest_key(b.nbest(fst, n=4))
    first = bits(b.posteriors(fst, 0.3, 1.5, 1e-3))
    for _ in range(2):
        assert bits(b.posteriors(fst, 0.3, 1.5, 1e-3)) == first
    assert nbest_key(b.nbest(fst, n=4)) == nb
    b.posteriors(fst)
    lats2, best2 = b.lattice(fst, lattice_beam=4.0)
    assert best2.tobytes() == best.tobytes() and all(same_records(x, y) for x, y in zip(lats, lats2))
    b.posteriors(fst)
    hyps2, wts2 = b.decode(fst)
    assert hyps2 == hyps and wts2.tobytes() == wts.tobytes()
    b.close()
    fst.close()
    am.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["loop", "eps"])
def test_online_posteriors_equal_batch_posteriors_for_any_split(ctx, kind):
    am, fst, _, _ = make_model(ctx, kind)
    lens = LENS + [0]
    b, rows = batch_of(ctx, am, lens, seed=500)
    b.lattice(fst, lattice_beam=4.0)
    want = bits(b.posteriors(fst, 0.3, 1.5, 1e-3))
    b.close()
    T = max(r.shape[0] for r in rows)
    for k in (1, 7, T):
        dec = pk.Decoder(ctx, am, fst, len(lens))
        dec.set_lattice(4.0, max_frames=T)
        with pytest.raises(pk.PkbError):
            dec.posteriors()    # no finish yet
        decode_in_splits(dec, rows, k)
        assert bits(dec.posteriors(0.3, 1.5, 1e-3)) == want, (kind, k)
        dec.close()
    fst.close()
    am.close()


def check_attached_stream_posteriors():
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
        got = bits(dec.posteriors(1.0, 1.0, 1e-3))
        rows = stream_rows(st, pcm, chunk, rows=True)
        dec.finish()
        ref.advance(np.stack(rows))
        ref.finish()
        assert got == bits(ref.posteriors(1.0, 1.0, 1e-3)) == bits(dec.posteriors(1.0, 1.0, 1e-3)), rep
        assert all(len(f) for f in dec.posteriors()[2])
    for o in (st, dec, ref, fst, am):
        o.close()
    ctx.close()


@pytest.mark.gpu
def test_attached_stream_posteriors():
    check_attached_stream_posteriors()


@pytest.mark.gpu
def test_attached_stream_posteriors_eager():
    run_child("import test_gpu_posteriors as t\nt.check_attached_stream_posteriors()\nprint('CHILD OK')",
              PKB_STREAM_GRAPH="0")


@pytest.mark.gpu
def test_arc_overflow_fails_only_its_utterance(ctx):
    am, fst, graph, tid2pdf = make_model(ctx, "loop")
    b, rows = batch_of(ctx, am, LENS)
    n_log = [host_lattice(graph, tid2pdf, r, lattice_beam=4.0)[2] for r in rows]
    big = int(np.argmax(n_log))
    lats, best = b.lattice(fst, lattice_beam=4.0, max_arcs=n_log[big] - 1)
    tot = np.zeros(len(rows))
    npost = np.zeros(len(rows), np.int64)
    assert ctx.lib.pkb_batch_posteriors(b.h, fst.h, 1.0, 1.0, 0.0, tot.ctypes.data, npost.ctypes.data) == 0
    assert npost[big] == -4 and math.isnan(tot[big])
    got = b.posteriors(fst)
    assert got[1][big] is None and got[2][big] is None
    check_against_host(got, lats, best, graph, tid2pdf, (1.0, 1.0), 0.0, "overflow")
    assert all(got[2][u] is not None for u in range(len(rows)) if u != big)
    assert any(len(got[2][u]) for u in range(len(rows)) if u != big)
    b.close()
    fst.close()
    am.close()


def eps_cycle_model(ctx):
    """make_model's "eps" kind with a two-state epsilon cycle hub -> X -> hub (no labels)."""
    rng = np.random.default_rng(2)
    P = 96
    layers = formats.make_dnn(rng, 440, 96, 2, P)
    layers[-2] = ("linear", (layers[-2][1] * 3.0).astype(np.float32), layers[-2][2])
    prior = rng.uniform(0.5, 1.5, P).astype(np.float32)
    prior /= prior.sum()
    (S, start, finals, arcs), tid2pdf = eps_graph(10, 3, P)
    graph = (S + 1, start, finals, arcs + [(1, S, 0, 0, 0.3), (S, 1, 0, 0, 0.4)])
    am = pk.AcousticModel(ctx, pk.PREC_BF16X3).from_layers(layers, prior, 5, 5, tid2pdf=tid2pdf)
    return am, pk.Fst(ctx, graph=graph)


@pytest.mark.gpu
def test_epsilon_cycle_fails_each_affected_utterance(ctx):
    am, fst = eps_cycle_model(ctx)
    b, rows = batch_of(ctx, am, [16000, 8000, 0])
    lats, best = b.lattice(fst, lattice_beam=INF)
    tot = np.zeros(3)
    npost = np.zeros(3, np.int64)
    assert ctx.lib.pkb_batch_posteriors(b.h, fst.h, 1.0, 1.0, 0.0, tot.ctypes.data, npost.ctypes.data) == 0
    got = b.posteriors(fst)
    for u, lat in enumerate(lats):
        cyc = host_posteriors(lat, lattice_T(lat), 0, {}, [0] * 100, num_states=fst_states(lat))[0] == -8
        assert cyc, u
        assert npost[u] == -8 and math.isnan(tot[u])
        assert len(got[1][u]) == len(lat) and np.isnan(got[1][u]).all() and got[2][u] is None
    assert all(x for x in b.nbest(fst, n=4))
    b.close()
    fst.close()
    am.close()


def fst_states(lat):
    return int(max(lat["src"].max(), lat["dst"].max())) + 1


@pytest.mark.gpu
def test_invalid_uses_are_rejected(ctx):
    am, fst, _, _ = make_model(ctx, "loop")
    am2, fst2, _, _ = make_model(ctx, "loop")
    b, _ = batch_of(ctx, am, [16000, 8000])
    with pytest.raises(pk.PkbError):
        b.posteriors(fst)                 # no lattice yet
    tot = np.zeros(2)
    npost = np.zeros(2, np.int64)
    assert ctx.lib.pkb_batch_posteriors_get(b.h, None, None) == 1   # before its call
    b.lattice(fst, lattice_beam=4.0)
    assert ctx.lib.pkb_batch_posteriors_get(b.h, None, None) == 1   # before its call on this lattice
    with pytest.raises(pk.PkbError):
        b.posteriors(fst2)                # another graph
    nan = float("nan")
    for a, g, m in ((0.0, 1.0, 0.0), (-1.0, 1.0, 0.0), (nan, 1.0, 0.0), (INF, 1.0, 0.0), (-INF, 1.0, 0.0),
                    (1.0, -0.5, 0.0), (1.0, nan, 0.0), (1.0, INF, 0.0),
                    (1.0, 1.0, -0.1), (1.0, 1.0, 1.5), (1.0, 1.0, nan)):
        with pytest.raises(pk.PkbError):
            b.posteriors(fst, a, g, m)
    for i in range(2):
        ptrs = [0 if j == i else o.ctypes.data for j, o in enumerate((tot, npost))]
        assert ctx.lib.pkb_batch_posteriors(b.h, fst.h, 1.0, 1.0, 0.0, *ptrs) == 1
    assert ctx.lib.pkb_batch_posteriors(b.h, fst.h, 1.0, 0.0, 1.0, tot.ctypes.data, npost.ctypes.data) == 0
    assert ctx.lib.pkb_batch_posteriors_get(b.h, None, None) == 0   # both outputs may be NULL
    before = bits(b.posteriors(fst))
    with pytest.raises(pk.PkbError):
        b.lattice(fst, lattice_beam=-1.0)   # refused before it touches the latest lattice
    assert bits(b.posteriors(fst)) == before
    b.close()
    dec = pk.Decoder(ctx, am, fst, 2)
    with pytest.raises(pk.PkbError):
        dec.posteriors()                  # before the first finish
    assert ctx.lib.pkb_decoder_posteriors_get(dec.h, None, None) == 1
    rows = np.zeros((2, 4, am.num_pdfs()), np.float32)
    dec.advance(rows)
    dec.finish()
    with pytest.raises(pk.PkbError):
        dec.posteriors()                  # that finish ran without lattices
    dec.set_lattice(4.0)
    dec.advance(rows)
    dec.finish()
    assert ctx.lib.pkb_decoder_posteriors_get(dec.h, None, None) == 1   # before its call
    assert len(dec.posteriors()[1]) == 2
    for a, g, m in ((0.0, 1.0, 0.0), (1.0, -1.0, 0.0), (1.0, 1.0, 2.0)):
        with pytest.raises(pk.PkbError):
            dec.posteriors(a, g, m)
    for i in range(2):
        ptrs = [0 if j == i else o.ctypes.data for j, o in enumerate((tot, npost))]
        assert ctx.lib.pkb_decoder_posteriors(dec.h, 1.0, 1.0, 0.0, *ptrs) == 1
    dec.advance(rows)
    with pytest.raises(pk.PkbError):
        dec.posteriors()                  # after an advance
    assert ctx.lib.pkb_decoder_posteriors_get(dec.h, None, None) == 1
    dec.close()
    fst2.close()
    am2.close()
    fst.close()
    am.close()


@pytest.mark.gpu
def test_posterior_cycles_do_not_leak(ctx):
    import torch
    am, fst, _, _ = make_model(ctx, "loop_big")
    pcm = coloured(7, 16000)

    def cycle():
        b = pk.Batch(ctx, [16000, 16000], synth_global_cmvn(), am, prob_scale=0.1)
        b.set_pcm(np.ascontiguousarray(np.concatenate([pcm, pcm]), np.int16))
        b.run(pk.STAGE_ALL)
        b.lattice(fst, lattice_beam=4.0)
        tot, arcs, frames = b.posteriors(fst, min_post=1e-3)
        assert np.isfinite(tot).all() and all(len(f) for f in frames)
        b.close()

    cycle()
    before = torch.cuda.mem_get_info(0)[0]
    for _ in range(20):
        cycle()
    assert before - torch.cuda.mem_get_info(0)[0] <= MARGIN
    fst.close()
    am.close()
