"""Speed and words of max-active pruning (pkb_batch_set_max_active) on a graph whose beam holds
thousands of tokens: an epsilon-hub word loop of 1,300 words x 3 HMM states (5,202 states, 10,401
arcs; table kernel with global tables), config-3 net (6x1024 -> 3000 pdfs) in fp16r, 128 synthetic
utterances of 10 s, beam 16, max_tokens = the state count (a frame can hold no more tokens, so the
unpruned search never overflows). For max_active 0 (off), 4000, 1000 and 250 it reports
pkb_batch_decode and pkb_batch_lattice (lattice beam 8) times -- host clock around each synchronous
call, median over repetitions that alternate the two calls, after one warm-up of both -- the
utterances whose words equal the unpruned search's, and failures. The 40-word loop of
tools/decode_demo.py (121 states, dense kernel) runs at 0 and 100. An unpruned lattice call on the
hub graph can take tens of seconds: once one passes --slow seconds, its remaining repetitions are
skipped (the run says how many it took).
Usage on a B200: python tools/max_active_bench.py [--reps 3] [--out profiles/max_active_bench.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pocketkaldi_b200 as pk  # noqa: E402
from pocketkaldi_b200 import formats  # noqa: E402
from pocketkaldi_b200.synth import synth_global_cmvn  # noqa: E402
from tools.decode_demo import word_loop_graph  # noqa: E402

P = 3000


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, universal_newlines=True, check=True).stdout
    name, limit = [x.strip() for x in q.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": limit}


def hub_graph(n_words, n_hmm, num_pdfs):
    """Word loop through an epsilon hub: start -eps-> hub -> word entry (emitting); word end -eps->
    tail -eps(word label)-> hub. Word ends and the hub are final. The labels sit on the arcs into the
    hub, so a frame adds one word record (the hub's token), not one per word entered."""
    arcs, tid2pdf = [], [0]
    hub = 1
    state_of = lambda w, s: 2 + n_words + w * n_hmm + s
    tid = 1
    enter = {}
    for w in range(n_words):
        for s in range(n_hmm):
            pdf = (w * n_hmm + s) % num_pdfs
            arcs.append((state_of(w, s), state_of(w, s), tid, 0, 0.05))
            tid2pdf.append(pdf)
            enter[(w, s)] = tid + 1
            tid2pdf.append(pdf)
            tid += 2
    arcs.append((0, hub, 0, 0, 0.1))
    for w in range(n_words):
        arcs.append((hub, state_of(w, 0), enter[(w, 0)], 0, 0.2 + 0.001 * w))
        for s in range(1, n_hmm):
            arcs.append((state_of(w, s - 1), state_of(w, s), enter[(w, s)], 0, 0.1))
        arcs.append((state_of(w, n_hmm - 1), 2 + w, 0, 0, 0.05))
        arcs.append((2 + w, hub, 0, w + 1, 0.02))
    finals = {state_of(w, n_hmm - 1): 0.3 for w in range(n_words)}
    finals[hub] = 0.0
    return (2 + n_words + n_words * n_hmm, 0, finals, arcs), tid2pdf


def lattice_counts(b, fst, max_tokens):
    n = len(b.num_samples)
    na = np.zeros(n, np.int64)
    best = np.zeros(n, np.float64)
    pk.binding._check(b.ctx.lib.pkb_batch_lattice(b.h, fst.h, 0.0, 8.0, max_tokens, 0, na.ctypes.data,
                                                  best.ctypes.data))
    return na


def measure(ctx, layers, prior, graph, tid2pdf, values, reps, slow, utts):
    max_tokens = graph[0]
    am = pk.AcousticModel(ctx, pk.PREC_FP16R).from_layers(layers, prior, 5, 5, tid2pdf=np.asarray(tid2pdf, np.int32))
    fst = pk.Fst(ctx, graph=graph)
    b = pk.Batch(ctx, [160000] * utts, synth_global_cmvn(), am, prob_scale=0.1)
    b.synth_pcm(1234, 0)
    b.run(pk.STAGE_ALL | pk.STAGE_NO_FEATS)
    ctx.sync()
    b.set_max_active(values[-1])   # warm-up of both calls and their buffers, at the cheapest setting
    b.decode(fst, max_tokens=max_tokens)
    lattice_counts(b, fst, max_tokens)
    runs, ref = [], None
    for ma in values:
        b.set_max_active(ma)
        t_dec, t_lat = [], []
        for _ in range(reps):
            t0 = time.perf_counter()
            hyps, _ = b.decode(fst, max_tokens=max_tokens)
            t1 = time.perf_counter()
            t_dec.append(t1 - t0)
            if not t_lat or max(t_lat) < slow:
                na = lattice_counts(b, fst, max_tokens)
                t_lat.append(time.perf_counter() - t1)
        if ref is None:
            ref = hyps
        run = {"graph": "%d states, %d arcs" % (graph[0], len(graph[3])), "max_active": ma, "utts": utts,
               "decode_ms": float(np.median(t_dec)) * 1e3, "lattice_ms": float(np.median(t_lat)) * 1e3,
               "decode_ms_all": [x * 1e3 for x in t_dec], "lattice_ms_all": [x * 1e3 for x in t_lat],
               "words_equal_to_unpruned": int(sum(h == r for h, r in zip(hyps, ref))),
               "words_per_utt": float(np.mean([len(h) for h in hyps if h is not None] or [0])),
               "decode_failed": int(sum(h is None for h in hyps)), "lattice_failed": int(np.sum(na < 0)),
               "lattice_arcs_per_utt": float(np.maximum(na, 0).mean())}
        print(json.dumps(run), flush=True)
        runs.append(run)
    for o in (b, fst, am):
        o.close()
    return runs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--utts", type=int, default=128)
    ap.add_argument("--slow", type=float, default=20.0, help="seconds after which a lattice call is not repeated")
    ap.add_argument("--out", default="profiles/max_active_bench.json")
    args = ap.parse_args()
    ctx = pk.Context(0)
    rng = np.random.default_rng(0)
    layers = formats.make_dnn(rng, 440, 1024, 6, P)
    prior = np.full(P, 1.0 / P, np.float32)
    res = {"card": card(), "precision": "fp16r", "utterance_seconds": 10.0, "beam": 16.0, "lattice_beam": 8.0}
    graph, tid2pdf = hub_graph(1300, 3, P)
    res["hub"] = measure(ctx, layers, prior, graph, tid2pdf, [0, 4000, 1000, 250], args.reps, args.slow, args.utts)
    graph, tid2pdf = word_loop_graph(40, 3, P)
    res["loop40"] = measure(ctx, layers, prior, graph, tid2pdf, [0, 100], args.reps, args.slow, args.utts)
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card"]}))
    ctx.close()


if __name__ == "__main__":
    main()
