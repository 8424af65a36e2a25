"""Cost of best paths with alignments over lattices (pkb_batch_best_path, pkb_decoder_best_path) next to
the lattice call they follow: config-3 net (6x1024 -> 3000 pdfs) in the default precision (fp16r), 10 s
synthetic utterances, the word-loop graphs of tools/lattice_bench.py (40 words, dense kernel; 180 words,
table kernel). The calls are synchronous, so a host clock around each call is its time; they alternate
over the repetitions after one warm-up of each shape, and the medians are reported. A best-path time
includes its _get call (words, word times and alignments to host memory).
  - 40-word loop, 128 and 1024 utterances at lattice beams 4 and 8, scales of 1 and no penalty;
  - 180-word loop, 128 utterances at lattice beam 4;
  - 64 streams of the online decoder on the 40-word loop: pkb_decoder_finish + pkb_decoder_best_path
    against the copy of every lattice record to pageable host memory that it replaces;
  - a scoring sweep over 128 utterances of the 40-word loop at lattice beam 8: LMWT 7..17 (acoustic
    scale 1 / LMWT) x word insertion penalty 0 / 0.5 / 1, 33 best paths, against the copy of every
    lattice record to pageable host memory, timed in the same run.
Usage on a B200: python tools/best_path_bench.py [--reps 3] [--out profiles/best_path_bench.json]"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pocketkaldi_b200 as pk  # noqa: E402
from pocketkaldi_b200 import formats  # noqa: E402
from pocketkaldi_b200.synth import synth_global_cmvn  # noqa: E402
from tools.decode_demo import word_loop_graph  # noqa: E402
from tools.lattice_bench import card, lattice_counts  # noqa: E402
from tools.nbest_bench import timed  # noqa: E402

SWEEP = [(1.0 / lmwt, 1.0, wip) for lmwt in range(7, 18) for wip in (0.0, 0.5, 1.0)]


def summary(res, frames):
    ok = [r for r in res if r is not None]
    return {"failed": len(res) - len(ok), "words": int(sum(len(r[3]) for r in ok)),
            "aligned_frames": int(sum(len(r[5]) for r in ok)), "frames": frames,
            "finite_costs": int(sum(np.isfinite(r[0]) for r in ok))}


def batch_runs(ctx, layers, prior, reps):
    runs = []
    for words, sizes, beams in ((40, (128, 1024), (4.0, 8.0)), (180, (128,), (4.0,))):
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
                lattice_counts(b, fst, lb, 0)
                b.best_path(fst)   # warm-up of this shape
                t_lat, t_bp = [], []
                for _ in range(reps):
                    dt, na = timed(lambda: lattice_counts(b, fst, lb, 0))
                    t_lat.append(dt)
                    dt, res = timed(lambda: b.best_path(fst))
                    t_bp.append(dt)
                run = {"graph": "%d-word loop (%d states, %d arcs)" % (words, graph[0], len(graph[3])),
                       "utts": utts, "lattice_beam": lb, "kept_arcs": int(na[na >= 0].sum()),
                       "kept_arcs_per_frame": float(na[na >= 0].sum()) / frames,
                       "lattice_ms": float(np.median(t_lat)) * 1e3, "best_path_ms": float(np.median(t_bp)) * 1e3,
                       "lattice_ms_all": [x * 1e3 for x in t_lat], "best_path_ms_all": [x * 1e3 for x in t_bp]}
                run.update(summary(res, frames))
                print(json.dumps(run), flush=True)
                runs.append(run)
                if words == 40 and utts == 128 and lb == 8.0:
                    sweep = sweep_run(b, fst, reps, frames)
            b.close()
        fst.close()
        am.close()
    return runs, sweep


def sweep_run(b, fst, reps, frames):
    """The 33 (LMWT, WIP) best paths of a scoring sweep against one copy of the records."""
    def sweep():
        return [b.best_path(fst, *s) for s in SWEEP]

    def copy():   # every record to pageable host memory, as a caller without best paths takes them
        arcs = np.empty(max(int(na[na >= 0].sum()), 1), pk.LATTICE_ARC_DTYPE)
        pk.binding._check(b.ctx.lib.pkb_batch_lattice_get(b.h, arcs.ctypes.data))
        return arcs

    na = lattice_counts(b, fst, 8.0, 0)
    sweep()
    copy()
    t_sweep, t_copy = [], []
    for _ in range(reps):
        dt, res = timed(sweep)
        t_sweep.append(dt)
        dc, _ = timed(copy)
        t_copy.append(dc)
    run = {"graph": "40-word loop", "utts": len(b.num_samples), "lattice_beam": 8.0, "points": len(SWEEP),
           "lmwt": [7, 17], "wip": [0.0, 0.5, 1.0],
           "sweep_ms": float(np.median(t_sweep)) * 1e3, "sweep_ms_all": [x * 1e3 for x in t_sweep],
           "record_copy_ms": float(np.median(t_copy)) * 1e3, "record_copy_ms_all": [x * 1e3 for x in t_copy],
           "record_bytes": int(na[na >= 0].sum()) * pk.LATTICE_ARC_DTYPE.itemsize,
           "words_per_point": [int(sum(len(r[3]) for r in p if r is not None)) for p in res]}
    run.update(summary(res[0], frames))
    print(json.dumps(run), flush=True)
    return run


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
    t_fin, t_bp, t_copy = [], [], []
    for rep in range(reps + 1):
        for t0 in range(0, ll.shape[1], 16):
            dec.advance(ll[:, t0:t0 + 16])
        dt, _ = timed(dec.finish)
        dp, res = timed(dec.best_path)
        dc, (lats, _) = timed(dec.lattice)   # every record to pageable host memory
        if rep:
            t_fin.append(dt)
            t_bp.append(dp)
            t_copy.append(dc)
    na = np.array([-1 if x is None else len(x) for x in lats], np.int64)
    run = {"graph": "40-word loop", "streams": S, "frames_per_stream": int(ll.shape[1]), "lattice_beam": 4.0,
           "finish_ms": float(np.median(t_fin)) * 1e3, "best_path_ms": float(np.median(t_bp)) * 1e3,
           "record_copy_ms": float(np.median(t_copy)) * 1e3,
           "record_bytes": int(na[na >= 0].sum()) * pk.LATTICE_ARC_DTYPE.itemsize}
    run.update(summary(res, S * int(ll.shape[1])))
    print(json.dumps(run), flush=True)
    dec.close()
    fst.close()
    am.close()
    return run


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="profiles/best_path_bench.json")
    args = ap.parse_args()
    ctx = pk.Context(0)
    rng = np.random.default_rng(0)
    P = 3000
    layers = formats.make_dnn(rng, 440, 1024, 6, P)
    prior = np.full(P, 1.0 / P, np.float32)
    res = {"card": card(), "precision": "fp16r", "utterance_seconds": 10.0}
    res["runs"], res["sweep"] = batch_runs(ctx, layers, prior, args.reps)
    res["online"] = online_run(ctx, layers, prior, args.reps)
    res["card_after"] = card()
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card"]}))
    ctx.close()


if __name__ == "__main__":
    main()
