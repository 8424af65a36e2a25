"""Cost of N-best lists over lattices (pkb_batch_nbest, pkb_decoder_nbest) next to the lattice call they
follow: config-3 net (6x1024 -> 3000 pdfs) in the default precision (fp16r), 10 s synthetic utterances,
the word-loop graphs of tools/lattice_bench.py (40 words, dense kernel; 180 words, table kernel).
Both calls are synchronous, so a host clock around each call is its time; they alternate over the
repetitions after one warm-up of each shape, and the medians are reported.
  - 40-word loop, 128 and 1024 utterances, n = 1 / 10 / 100 at lattice beams 4 and 8;
  - 180-word loop, 128 utterances, n = 10 at lattice beam 4;
  - 64 streams of the online decoder on the 40-word loop: pkb_decoder_finish + pkb_decoder_nbest
    against the copy of every lattice record to pageable host memory that it replaces.
Usage on a B200: python tools/nbest_bench.py [--reps 5] [--out profiles/nbest_bench.json]"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pocketkaldi_b200 as pk  # noqa: E402
from pocketkaldi_b200 import formats  # noqa: E402
from pocketkaldi_b200.synth import synth_global_cmvn  # noqa: E402
from tools.decode_demo import word_loop_graph  # noqa: E402
from tools.lattice_bench import card, lattice_counts  # noqa: E402


def timed(f):
    t0 = time.perf_counter()
    r = f()
    return time.perf_counter() - t0, r


def batch_runs(ctx, layers, prior, reps):
    runs = []
    for words, sizes, ns, beams in ((40, (128, 1024), (1, 10, 100), (4.0, 8.0)), (180, (128,), (10,), (4.0,))):
        graph, tid2pdf = word_loop_graph(words, 3, 3000)
        am = pk.AcousticModel(ctx, pk.PREC_FP16R).from_layers(layers, prior, 5, 5,
                                                              tid2pdf=np.asarray(tid2pdf, np.int32))
        fst = pk.Fst(ctx, graph=graph)
        for utts in sizes:
            b = pk.Batch(ctx, [160000] * utts, synth_global_cmvn(), am, prob_scale=0.1)
            b.synth_pcm(1234, 0)
            b.run(pk.STAGE_ALL | pk.STAGE_NO_FEATS)
            ctx.sync()
            frames = int(b.num_frames.sum())
            for lb in beams:
                for n in ns:
                    lattice_counts(b, fst, lb, 0)
                    b.nbest(fst, n=n)   # warm-up of this shape
                    t_lat, t_nb = [], []
                    for _ in range(reps):
                        dt, na = timed(lambda: lattice_counts(b, fst, lb, 0))
                        t_lat.append(dt)
                        dt, lists = timed(lambda: b.nbest(fst, n=n))
                        t_nb.append(dt)
                    run = {"graph": "%d-word loop (%d states, %d arcs)" % (words, graph[0], len(graph[3])),
                           "utts": utts, "frames": frames, "lattice_beam": lb, "n": n,
                           "kept_arcs_per_frame": float(na[na >= 0].sum()) / frames,
                           "lattice_ms": float(np.median(t_lat)) * 1e3, "nbest_ms": float(np.median(t_nb)) * 1e3,
                           "lattice_ms_all": [x * 1e3 for x in t_lat], "nbest_ms_all": [x * 1e3 for x in t_nb],
                           "failed": int(sum(x is None for x in lists)),
                           "mean_entries": float(np.mean([len(x) for x in lists if x is not None]))}
                    print(json.dumps(run), flush=True)
                    runs.append(run)
            b.close()
        fst.close()
        am.close()
    return runs


def online_run(ctx, layers, prior, reps):
    """64 streams of 10 s rows on the 40-word loop, fed in 16-frame advances."""
    graph, tid2pdf = word_loop_graph(40, 3, 3000)
    am = pk.AcousticModel(ctx, pk.PREC_FP16R).from_layers(layers, prior, 5, 5, tid2pdf=np.asarray(tid2pdf, np.int32))
    fst = pk.Fst(ctx, graph=graph)
    S = 64
    b = pk.Batch(ctx, [160000] * S, synth_global_cmvn(), am, prob_scale=0.1)
    b.synth_pcm(99, 0)
    b.run(pk.STAGE_ALL)
    ll = b.get(pk.BUF_LOGLIK).reshape(S, -1, 3000)
    b.close()
    dec = pk.Decoder(ctx, am, fst, S)
    dec.set_lattice(4.0, max_frames=ll.shape[1])
    t_fin, t_nb, t_copy = [], [], []
    for rep in range(reps + 1):
        for t0 in range(0, ll.shape[1], 16):
            dec.advance(ll[:, t0:t0 + 16])
        dt, _ = timed(dec.finish)
        dn, lists = timed(lambda: dec.nbest(n=10))
        dc, (lats, _) = timed(dec.lattice)   # every record to pageable host memory
        if rep:
            t_fin.append(dt)
            t_nb.append(dn)
            t_copy.append(dc)
    run = {"graph": "40-word loop", "streams": S, "frames_per_stream": int(ll.shape[1]), "lattice_beam": 4.0,
           "n": 10, "finish_ms": float(np.median(t_fin)) * 1e3, "nbest_ms": float(np.median(t_nb)) * 1e3,
           "record_copy_ms": float(np.median(t_copy)) * 1e3,
           "record_bytes": int(sum(len(x) for x in lats if x is not None)) * pk.LATTICE_ARC_DTYPE.itemsize,
           "failed": int(sum(x is None for x in lists))}
    print(json.dumps(run), flush=True)
    dec.close()
    fst.close()
    am.close()
    return run


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="profiles/nbest_bench.json")
    args = ap.parse_args()
    ctx = pk.Context(0)
    rng = np.random.default_rng(0)
    P = 3000
    layers = formats.make_dnn(rng, 440, 1024, 6, P)
    prior = np.full(P, 1.0 / P, np.float32)
    res = {"card": card(), "precision": "fp16r", "utterance_seconds": 10.0,
           "runs": batch_runs(ctx, layers, prior, args.reps), "online": online_run(ctx, layers, prior, args.reps)}
    res["card_after"] = card()
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card"]}))
    ctx.close()


if __name__ == "__main__":
    main()
