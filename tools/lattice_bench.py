"""Cost of lattice output (pkb_batch_lattice) next to the plain batch search (pkb_batch_decode) on
the same batch: config-3 net (6x1024 -> 3000 pdfs) in the default precision (fp16r), 10 s synthetic
utterances, two word-loop graphs of tools/decode_demo.py: 40 words (1,840 arcs, dense kernel) and
180 words (table kernel, global tables). Both calls are synchronous, so a host clock around each
call is its time; the two are alternated over the repetitions.
Per graph and batch size it reports: decode and lattice times (median over repetitions); kept arcs
per frame at lattice beams 2, 4, 8 and +inf; the largest unpruned log of an utterance (the least
max_arcs with no overflow, by bisection on the 128-utterance batch) and the device bytes of the log
at the default max_arcs ((frames + 1) x graph arcs). The 180-word loop keeps ~33 k arcs per frame
inside the beam, 267 MB of log per 10 s utterance: it runs at 128 utterances only, since 1024 of
them would need 274 GB.
Usage on a B200: python tools/lattice_bench.py [--reps 5] [--out profiles/lattice_bench.json]"""
import argparse
import json
import math
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

FRAMES = 998  # frames of a 10 s utterance


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, universal_newlines=True, check=True).stdout
    name, limit = [x.strip() for x in q.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": limit}


def lattice_counts(b, fst, lattice_beam, max_arcs):
    n = len(b.num_samples)
    na = np.zeros(n, np.int64)
    best = np.zeros(n, np.float64)
    pk.binding._check(b.ctx.lib.pkb_batch_lattice(b.h, fst.h, 0.0, lattice_beam, 0, max_arcs, na.ctypes.data,
                                                  best.ctypes.data))
    return na


def max_log(b, fst):
    """Least max_arcs for which no utterance of the batch overflows its log (a narrow lattice beam
    keeps the probes cheap: the log does not depend on it)."""
    lo, hi = 0, 1 << 21
    while np.any(lattice_counts(b, fst, 1e-3, hi) == -4):
        lo, hi = hi, hi * 2
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if np.any(lattice_counts(b, fst, 1e-3, mid) == -4):
            lo = mid
        else:
            hi = mid
    return hi


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="profiles/lattice_bench.json")
    args = ap.parse_args()
    ctx = pk.Context(0)
    rng = np.random.default_rng(0)
    P = 3000
    layers = formats.make_dnn(rng, 440, 1024, 6, P)
    prior = np.full(P, 1.0 / P, np.float32)
    res = {"card": card(), "precision": "fp16r", "utterance_seconds": 10.0, "runs": []}
    for words in (40, 180):
        graph, tid2pdf = word_loop_graph(words, 3, P)
        am = pk.AcousticModel(ctx, pk.PREC_FP16R).from_layers(layers, prior, 5, 5,
                                                              tid2pdf=np.asarray(tid2pdf, np.int32))
        fst = pk.Fst(ctx, graph=graph)
        max_arcs = (FRAMES + 1) * len(graph[3])  # the default of pkb_batch_lattice
        for n in (128, 1024):
            log_bytes = n * max_arcs * 8
            if log_bytes > (100 << 30):
                res["runs"].append({"graph": "%d-word loop" % words, "utts": n, "not_run": True,
                                    "log_bytes": log_bytes})
                continue
            b = pk.Batch(ctx, [160000] * n, synth_global_cmvn(), am, prob_scale=0.1)
            b.synth_pcm(1234, 0)
            b.run(pk.STAGE_ALL | pk.STAGE_NO_FEATS)
            ctx.sync()
            frames = int(b.num_frames.sum())
            assert int(b.num_frames.max()) == FRAMES
            b.decode(fst)
            lattice_counts(b, fst, 8.0, 0)  # warm-up of both paths and of the buffers
            t_dec, t_lat = [], []
            for _ in range(args.reps):
                t0 = time.perf_counter()
                hyps, _ = b.decode(fst)
                t1 = time.perf_counter()
                na = lattice_counts(b, fst, 8.0, 0)
                t2 = time.perf_counter()
                t_dec.append(t1 - t0)
                t_lat.append(t2 - t1)
            kept = {}
            for lb in (2.0, 4.0, 8.0, math.inf):
                na = lattice_counts(b, fst, lb, 0)
                kept["inf" if lb == math.inf else str(lb)] = {
                    "kept_arcs_per_frame": float(na[na >= 0].sum()) / frames, "failed": int(np.sum(na < 0))}
            run = {
                "graph": "%d-word loop (%d states, %d arcs)" % (words, graph[0], len(graph[3])),
                "utts": n, "frames": frames,
                "decode_ms": float(np.median(t_dec)) * 1e3, "lattice_ms": float(np.median(t_lat)) * 1e3,
                "decode_ms_all": [x * 1e3 for x in t_dec], "lattice_ms_all": [x * 1e3 for x in t_lat],
                "lattice_over_decode": float(np.median(t_lat) / np.median(t_dec)),
                "decode_failed": int(sum(h is None for h in hyps)),
                "kept": kept,
                "max_arcs": max_arcs, "log_bytes": log_bytes,
            }
            if n == 128:
                m = max_log(b, fst)
                run["max_unpruned_arcs_per_utt"] = m
                run["unpruned_arcs_per_frame_of_that_utt"] = m / float(b.num_frames.max())
                run["log_bytes_at_that_max_arcs"] = n * m * 8
            print(json.dumps(run), flush=True)
            res["runs"].append(run)
            b.close()
        fst.close()
        am.close()
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card"]}))
    ctx.close()


if __name__ == "__main__":
    main()
