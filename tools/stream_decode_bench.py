"""Push latency of the streaming pipeline with and without online GPU decoding (config-5 shape).

  python tools/stream_decode_bench.py [--steps 200] [--warmup 20] [--precision fp16r] [--out DIR]
  python tools/stream_decode_bench.py --profile-only [--out DIR]

64 streams x 2560-sample chunks (160 ms), the config-3 net (splice +-5 -> 6x1024 ReLU -> 3000
pdfs, random init) and the 40-word loop graph of tools/decode_demo.py (121 states, 1840 arcs: the
dense kernel). Three variants of the synchronous push are timed in one process, alternating push
by push, each on its own stream object with the same audio in pinned host buffers:
  (a) rows    pkb_stream_push_i16 with FP32 rows copied back, no decoder
  (b) decode  the same push with a decoder attached (rows and best-so-far copied back)
  (c) only    decode-only push (loglik_out NULL): only the best-so-far arrays cross PCIe
Latency is the host wall clock around the push (it ends in a stream synchronise). --profile-only
is the separate profiled run: decode-only pushes under torch.profiler (CUDA activities), giving the
advance kernel's device time per push; no latency is taken there. Prints one JSON object; with
--out also writes it (and the profiled run's trace) there.
"""

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

S, CHUNK, PDFS = 64, 2560, 3000


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, timeout=30).stdout.decode()
        name, limit = [x.strip() for x in q.strip().splitlines()[0].split(",")]
        return {"name": name, "power_limit": limit}
    except Exception as e:  # the measurement still stands; say what is missing
        return {"name": "unknown", "power_limit": "unknown (%s)" % e}


def stats(ms):
    ms = np.asarray(ms)
    return {"p50": float(np.percentile(ms, 50)), "p99": float(np.percentile(ms, 99)), "max": float(ms.max()),
            "mean": float(ms.mean()), "n": int(ms.size)}


def profile_advance(args, push, pin_in, audio):
    """Device time of the advance kernel per decode-only push, torch.profiler (CUPTI) over
    `--steps` pushes (at most 100) after the warm-up; kernels named viterbi_*, graph replays
    included."""
    from torch.profiler import ProfilerActivity, profile
    for k in range(args.warmup):
        pin_in.array[:] = audio[:, (k % 8) * CHUNK:((k % 8) + 1) * CHUNK]
        push("c_decode_only")
    n_prof = min(args.steps, 100)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for k in range(n_prof):
            pin_in.array[:] = audio[:, (k % 8) * CHUNK:((k % 8) + 1) * CHUNK]
            push("c_decode_only")
    kern = {}
    for e in prof.events():
        if "viterbi" in e.name:
            t = e.device_time if hasattr(e, "device_time") else e.cuda_time
            name = e.name[:e.name.find("(", e.name.index("viterbi"))].replace("(anonymous namespace)::", "")
            kern.setdefault(name, []).append(t)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        prof.export_chrome_trace(os.path.join(args.out, "stream_decode_trace.json"))
    return {"advance_kernel_us_per_push": sum(sum(v) for v in kern.values()) / n_prof,
            "advance_kernels_profiled": {k: len(v) for k, v in kern.items()},
            "advance_kernel_us_each": {k: float(np.mean(v)) for k, v in kern.items()},
            "profiled_pushes": n_prof}


def emit(args, res, name):
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, name), "w") as f:
            f.write(line + "\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--precision", default="fp16r")
    ap.add_argument("--out", default=None)
    ap.add_argument("--profile-only", action="store_true", help="the separate profiled run")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be positive and --warmup non-negative")

    import pocketkaldi_b200 as pk
    import tools.decode_demo as demo
    from pocketkaldi_b200 import formats
    from pocketkaldi_b200.binding import PinnedArray
    from pocketkaldi_b200.synth import synth_global_cmvn, synth_pcm

    prec = {"bf16": pk.PREC_BF16, "bf16x3": pk.PREC_BF16X3, "fp16": pk.PREC_FP16, "fp16x3": pk.PREC_FP16X3,
            "fp16c8": pk.PREC_FP16C8, "fp16r": pk.PREC_FP16R}[args.precision]
    info = card()
    ctx = pk.Context(0)
    layers = formats.make_dnn(np.random.default_rng(0), 440, 1024, 6, PDFS)
    graph, tid2pdf = demo.word_loop_graph(40, 3, PDFS)
    am = pk.AcousticModel(ctx, prec).from_layers(layers, np.full(PDFS, 1.0 / PDFS, np.float32), 5, 5,
                                                 tid2pdf=tid2pdf)
    fst = pk.Fst(ctx, graph=graph)
    g = synth_global_cmvn()
    n_chunks = args.warmup + args.steps
    audio = synth_pcm(1234, np.arange(S), CHUNK * 8)
    pin_in = PinnedArray((S, CHUNK), np.int16)

    names = ("a_rows", "b_rows_and_decode", "c_decode_only")
    streams, decs, outs = {}, {}, {}
    for nm in names:
        streams[nm] = pk.Stream(ctx, am, S, CHUNK, g, 0.1)
        outs[nm] = PinnedArray((S, streams[nm].max_frames, PDFS), np.float32)
        if nm != "a_rows":
            decs[nm] = pk.Decoder(ctx, am, fst, S)
            streams[nm].set_decoder(decs[nm])

    def push(nm):
        return streams[nm].push(pin_in.array, out=outs[nm].array, rows=nm != "c_decode_only")

    if args.profile_only:
        res = {"card": info, **profile_advance(args, push, pin_in, audio)}
        emit(args, res, "stream_decode_profile.json")
        ctx.close()
        return
    lat = {nm: [] for nm in names}
    frames = 0
    for k in range(n_chunks):
        pin_in.array[:] = audio[:, (k % 8) * CHUNK:((k % 8) + 1) * CHUNK]
        for nm in names[k % 3:] + names[:k % 3]:   # rotate the order push by push
            t0 = time.perf_counter()
            r = push(nm)
            t1 = time.perf_counter()
            if k >= args.warmup:
                lat[nm].append((t1 - t0) * 1e3)
            if nm == "a_rows" and k >= args.warmup:
                frames = r.shape[1]
    # the three variants decoded the same audio: their best-so-far results must agree
    pb, pc = decs["b_rows_and_decode"].partial(), decs["c_decode_only"].partial()
    agree = pb[0] == pc[0] and np.array_equal(pb[1], pc[1])

    mw = decs["c_decode_only"].max_words
    partial_bytes = S * (8 + 4 * mw + 4 + 4)
    row_bytes = S * frames * PDFS * 4
    res = {
        "card": info,
        "shape": {"streams": S, "chunk_samples": CHUNK, "frames_per_push": frames, "pdfs": PDFS,
                  "net": "440 -> 6x1024 ReLU -> 3000", "graph": "40-word loop, %d states, %d arcs" %
                  (graph[0], len(graph[3])), "precision": args.precision},
        "timing": "host wall clock around the synchronous push, %d pushes after %d warm-up, variants alternating"
                  % (args.steps, args.warmup),
        "latency_ms": {nm: stats(lat[nm]) for nm in names},
        "d2h_bytes_per_push": {"a_rows": row_bytes, "b_rows_and_decode": row_bytes + partial_bytes,
                               "c_decode_only": partial_bytes},
        "partials_agree_b_c": bool(agree),
        "best_so_far_words_stream0": pc[0][0],
    }
    for nm in names:
        streams[nm].close()
    for d in decs.values():
        d.close()
    emit(args, res, "stream_decode_bench.json")
    ctx.close()


if __name__ == "__main__":
    main()
