"""Cost of lattices in the online GPU decoder (pkb_decoder_set_lattice) on the shape of
tools/stream_decode_bench.py: 64 streams x 2560-sample chunks (160 ms), the config-3 net (splice +-5
-> 6x1024 ReLU -> 3000 pdfs, random init) in fp16r, decode-only pushes (loglik_out NULL).

  python tools/online_lattice_bench.py [--steps 200] [--warmup 20] [--reps 3] [--out profiles/online_lattice_bench.json]

Three measurements, all in one process on one card:
  push     40-word loop of tools/decode_demo.py (121 states, 1,840 arcs: the dense kernel). Two stream
           objects fed the same audio from the same pinned buffer, one decoder without and one with
           lattices (lattice beam 8); their decode-only pushes alternate push by push (order rotated).
           Latency: host wall clock around the synchronous push (it ends in a stream synchronise).
  finish   the same two decoders over 10 s utterances (63 decode-only pushes and a flush), at lattice
           beams 4 and 8: wall clock of pkb_decoder_finish (BestPath, with lattices also the backward
           pass, the record expansion and the copy of the per-stream counts), then of
           pkb_decoder_lattice_get (all records to pageable host memory) and its bytes.
  large    the 180-word loop (541 states, table kernel with global tables) at fewer streams and a
           stated max_arcs: push latency off / on and finish at lattice beam 8.
The lattice decoder's words and the other decoder's must agree (checked, reported).
"""

import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tools.stream_decode_bench import card, stats  # noqa: E402

CHUNK, PDFS = 2560, 3000
UTT_CHUNKS = 63   # 63 x 160 ms = 10.08 s, then a flush


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3, help="utterances timed per lattice beam")
    ap.add_argument("--streams", type=int, default=64)
    ap.add_argument("--large-streams", type=int, default=16)
    ap.add_argument("--large-max-arcs", type=int, default=40 << 20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "online_lattice_bench.json"))
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0 or args.reps < 1:
        ap.error("--steps and --reps must be positive, --warmup non-negative")

    import pocketkaldi_b200 as pk
    import tools.decode_demo as demo
    from pocketkaldi_b200 import formats
    from pocketkaldi_b200.binding import PinnedArray
    from pocketkaldi_b200.synth import synth_global_cmvn, synth_pcm

    info = card()
    ctx = pk.Context(0)
    layers = formats.make_dnn(np.random.default_rng(0), 440, 1024, 6, PDFS)
    g = synth_global_cmvn()
    res = {"card": info, "precision": "fp16r", "chunk_samples": CHUNK,
           "timing": "host wall clock around synchronous calls; off and on alternate call by call"}

    def run_graph(words, S, max_arcs, beams, steps, warmup, reps):
        graph, tid2pdf = demo.word_loop_graph(words, 3, PDFS)
        am = pk.AcousticModel(ctx, pk.PREC_FP16R).from_layers(layers, np.full(PDFS, 1.0 / PDFS, np.float32), 5, 5,
                                                               tid2pdf=tid2pdf)
        fst = pk.Fst(ctx, graph=graph)
        audio = synth_pcm(1234, np.arange(S), CHUNK * 8)
        pin = PinnedArray((S, CHUNK), np.int16)
        n_push = warmup + steps
        # frames the push phase puts in one utterance (16 per push), with room for the flush
        max_frames = max(n_push, UTT_CHUNKS) * 16 + 64
        st, dec = {}, {}
        for nm in ("off", "on"):
            st[nm] = pk.Stream(ctx, am, S, CHUNK, g, 0.1)
            dec[nm] = pk.Decoder(ctx, am, fst, S)
            if nm == "on":
                dec[nm].set_lattice(beams[-1], max_frames=max_frames, max_arcs=max_arcs)
            st[nm].set_decoder(dec[nm])

        def feed(k):
            pin.array[:] = audio[:, (k % 8) * CHUNK:((k % 8) + 1) * CHUNK]

        # ---- push latency, alternating
        lat = {"off": [], "on": []}
        for k in range(n_push):
            feed(k)
            for nm in (("off", "on") if k % 2 == 0 else ("on", "off")):
                t0 = time.perf_counter()
                st[nm].push(pin.array, rows=False)
                t1 = time.perf_counter()
                if k >= warmup:
                    lat[nm].append((t1 - t0) * 1e3)
        replays = {nm: st[nm].graph_replays() for nm in st}
        for nm in st:
            st[nm].flush(rows=False)
        ends = {nm: dec[nm].finish() for nm in dec}
        kept0 = dec["on"].lattice()
        out = {
            "graph": "%d-word loop, %d states, %d arcs" % (words, graph[0], len(graph[3])),
            "streams": S, "max_frames": max_frames,
            "max_arcs": max_arcs if max_arcs > 0 else min((max_frames + 1) * len(graph[3]), 2 ** 31 - 1),
            "push_ms": {nm: stats(lat[nm]) for nm in lat},
            "push_graph_replays": replays,
            "push_phase_frames_per_stream": n_push * 16,
            "push_phase_words_agree": ends["off"][0] == ends["on"][0],
            "push_phase_lattice_failed_streams": int(sum(x is None for x in kept0[0])),
        }
        # ---- finish of 10 s utterances
        out["finish"] = []
        lib = ctx.lib
        for lb in beams:
            dec["on"].set_lattice(lb, max_frames=max_frames, max_arcs=max_arcs)
            t_fin = {"off": [], "on": []}
            t_get, nbytes, kept, agree, failed = [], 0, 0, True, 0
            for r in range(reps + 1):   # the first utterance warms the new buffers up
                for k in range(UTT_CHUNKS):
                    feed(k + r)
                    for nm in ("off", "on"):
                        st[nm].push(pin.array, rows=False)
                fin = {}
                for nm in (("off", "on") if r % 2 == 0 else ("on", "off")):
                    st[nm].flush(rows=False)
                    t0 = time.perf_counter()
                    fin[nm] = dec[nm].finish()
                    t1 = time.perf_counter()
                    if r > 0:
                        t_fin[nm].append((t1 - t0) * 1e3)
                na = np.zeros(S, np.int64)
                best = np.zeros(S, np.float64)
                pk.binding._check(lib.pkb_decoder_lattice(dec["on"].h, na.ctypes.data, best.ctypes.data))
                total = int(np.maximum(na, 0).sum())
                arcs = np.empty(max(total, 1), pk.LATTICE_ARC_DTYPE)
                t0 = time.perf_counter()
                pk.binding._check(lib.pkb_decoder_lattice_get(dec["on"].h, C.c_void_p(arcs.ctypes.data)))
                t1 = time.perf_counter()
                if r > 0:
                    t_get.append((t1 - t0) * 1e3)
                    nbytes = total * pk.LATTICE_ARC_DTYPE.itemsize
                    kept = total
                    failed = int(np.sum(na < 0))
                agree = agree and fin["off"][0] == fin["on"][0] and fin["off"][1].tobytes() == fin["on"][1].tobytes()
            frames = (UTT_CHUNKS * CHUNK) // 160
            out["finish"].append({
                "lattice_beam": lb, "utterance_frames": frames,
                "finish_ms_off": stats(t_fin["off"]), "finish_ms_on": stats(t_fin["on"]),
                "lattice_get_ms": stats(t_get), "lattice_get_bytes": nbytes,
                "kept_arcs": kept, "kept_arcs_per_stream_frame": kept / float(S * frames),
                "failed_streams": failed, "words_and_weights_agree": bool(agree)})
        for nm in st:
            st[nm].close()
            dec[nm].close()
        fst.close()
        am.close()
        return out

    res["push_and_finish_40_word_loop"] = run_graph(40, args.streams, 0, (4.0, 8.0), args.steps, args.warmup,
                                                    args.reps)
    print(json.dumps(res["push_and_finish_40_word_loop"]), flush=True)
    res["large_180_word_loop"] = run_graph(180, args.large_streams, args.large_max_arcs, (8.0,),
                                           max(args.steps // 4, 10), min(args.warmup, 10), args.reps)
    print(json.dumps(res["large_180_word_loop"]), flush=True)
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"card": info, "out": args.out}))
    ctx.close()


if __name__ == "__main__":
    main()
