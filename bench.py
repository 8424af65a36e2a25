#!/usr/bin/env python
"""Benchmark of the acoustic front half: 16 kHz PCM -> fbank -> CMVN -> nnet log-likelihoods.

Contract (see the task statement): `python bench.py --gpus N --steps K --warmup W` prints ONE
JSON line on rank 0. A "step" is one pass of the hot path over one resident batch of synthetic
utterances. Default workload = BASELINE.json configs[2]: 4096 utterances x 10 s, splice +-5 ->
6 x 1024 ReLU DNN -> 3000 pdfs, tensor-core path, per GPU (weak scaling: every rank
processes its own 4096 utterances, no data-path collective; torch.distributed is used for the
barrier and the max-over-ranks time only). The reported `dtype` is DEFAULT_PRECISION: the
cheapest GEMM arithmetic that meets the parity bar (|dLL| <= 2e-2, argmax >= 99.9 %) on the
random-init nets BASELINE names -- tests/test_gpu_baseline_nets.py gates exactly this mode and
the line carries `parity_ok` for the run itself. The one-MMA modes (bf16, fp16) are reported in
`precision_modes` with their measured parity; they do not meet the bar (DESIGN.md section 1).

  value      frames/s with PCM already resident in HBM, CUDA events on the library's stream
  e2e        the same through the host-buffer API: pinned PCM H2D + compute + log-likelihood D2H
  roofline   dominant kernel (tcgen05 GEMM): algorithmic FLOPs / summed CUDA-event time of the
             GEMM launches in the timed region, against MEASURED_PEAKS.json
  cpu_baseline  the unmodified reference (oracle/_ref) timed on this host's cores (N=1 only)

`--impl reference` times the reference's own CPU path (all host threads) on the same config.
"""

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "acoustic frames/s (fbank+CMVN+nnet loglik)"
# The precision the headline is quoted in. tests/test_gpu_baseline_nets.py asserts the
# north_star parity bar for this mode on the config-3 and config-4 nets.
DEFAULT_PRECISION = "fp16r"
REFINE_MARGIN = float(os.environ.get("PKB_BENCH_REFINE_MARGIN", "0.02"))  # log-likelihood units; pkb_am_set_refine_margin
LL_TOL, ARGMAX_MIN, FEAT_TOL = 2e-2, 0.999, 1e-4
SAMPLES_10S = 160000
FRAMES_10S = 998
DUMP_LIMIT = 64 << 20  # bytes of all the files --dump-outputs writes

CONFIGS = {
    # name: (utts per GPU, hidden layers, width, pdfs, nnet?)
    "2": dict(utts=360, hidden=0, width=0, pdfs=0, nnet=False,
              name="config2: 1 h of 16 kHz audio in 10 s utterances, 40-dim fbank + CMVN only"),
    "3": dict(utts=4096, hidden=6, width=1024, pdfs=3000, nnet=True,
              name="config3: 4096 utts x 10 s, splice+-5 -> 6x1024 ReLU DNN -> 3000 pdfs"),
    "4": dict(utts=1024, hidden=7, width=2048, pdfs=8000, nnet=True,
              name="config4 shard: 1024 utts x 10 s per GPU, splice+-5 -> 7x2048 ReLU DNN -> 8000 pdfs"),
    "5": dict(utts=64, hidden=6, width=1024, pdfs=3000, nnet=True, stream=True,
              name="config5: 64 concurrent streams, 160 ms chunks (2560 samples), fbank+CMVN+6x1024->3000 nnet"),
}


for _k, _v in CONFIGS.items():
    _v["key"] = _k


def flops_per_frame(cfg):
    if not cfg["nnet"]:
        return 0
    h, w, p = cfg["hidden"], cfg["width"], cfg["pdfs"]
    return 2 * (440 * w + (h - 1) * w * w + w * p)


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm=d["hbm_gbs"], tensor_burst=d["bf16_tflops"],
                    tensor_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, tensor_burst=1590.0, tensor_sustained=1400.0, src="fallback")


def make_layers(cfg, seed=0):
    from pocketkaldi_b200 import formats
    rng = np.random.default_rng(seed)
    return formats.make_dnn(rng, 440, cfg["width"], cfg["hidden"], cfg["pdfs"])


class ClockSampler:
    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap,power.limit")

    def __init__(self, index):
        self.path = tempfile.mktemp(prefix="pkb_clocks_", suffix=".csv")
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.QUERY,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, pw, lim, reasons = [], [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 7:
                    continue
                try:
                    sm.append(float(f[0]))
                    mx.append(float(f[1]))
                except ValueError:
                    continue
                try:
                    pw.append(float(f[2]))
                except ValueError:
                    pw.append(0.0)
                try:
                    lim.append(float(f[7]))
                except (ValueError, IndexError):
                    pass
                for n, v in zip(names, f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            os.unlink(self.path)
        except OSError:
            pass
        if sm:
            # samples taken under load = those drawing at least 70 % of the highest power seen
            # (under a power cap the loaded clock is the LOWER one)
            loaded = [c for c, w in zip(sm, pw) if w >= 0.7 * max(pw)] or sm
            out["sm_mhz"] = float(np.median(loaded))
            out["sm_max_mhz"] = float(max(mx))
            out["power_w"] = float(np.median([w for w in pw if w >= 0.7 * max(pw)] or pw))
            if lim:
                out["power_limit_w"] = float(max(lim))
        out["reasons"] = sorted(reasons)
        out["samples"] = len(sm)
        return out


def dist_setup(n_gpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
    return rank, world, local, dist


def barrier(dist, local):
    if dist is not None:
        import torch
        dist.barrier(device_ids=[local])
        torch.cuda.synchronize()


def reduce_timing(dist, local, ms, frames):
    """(max over ranks of the device-timed ms, sum over ranks of frames)."""
    from pocketkaldi_b200 import sharding
    return sharding.reduce_timing(dist, ms, frames, device="cuda:%d" % local if dist else None)


# ----------------------------------------------------------------------------- reference arm
def write_reference_model(cfg, tmpdir):
    from pocketkaldi_b200 import formats
    from pocketkaldi_b200.synth import synth_global_cmvn
    layers = make_layers(cfg)
    prior = np.full(cfg["pdfs"], 1.0 / cfg["pdfs"], np.float32)
    tid2pdf = np.arange(-1, cfg["pdfs"], dtype=np.int32)
    tid2pdf[0] = 0
    return formats.write_model_dir(tmpdir, "bench", layers, prior, 5, 5, tid2pdf,
                                   cmvn_stats=synth_global_cmvn()), layers, prior


def time_reference(cfg, n_threads, n_utts, repeats):
    """Times the unmodified reference (oracle/_ref) on n_utts synthetic utterances."""
    from oracle.oracle import Reference
    from pocketkaldi_b200.synth import synth_pcm, synth_global_cmvn
    ref = Reference()
    g = synth_global_cmvn()
    pcm = synth_pcm(1234, np.arange(n_utts), SAMPLES_10S)
    am = None
    tmp = None
    if cfg["nnet"]:
        tmp = tempfile.TemporaryDirectory(prefix="pkb_bench_model_")
        conf, _, _ = write_reference_model(cfg, tmp.name)
        am = ref.am_load(conf)
    sec, frames, chk = ref.time_path(am, g, pcm, n_threads, repeats)
    if am:
        ref.am_free(am)
    if tmp:
        tmp.cleanup()
    return sec, frames, chk


def reference_sample_size(cfg, cores):
    # ~1.2 s per 10 s utterance per thread for the config-3 net, ~6 s for config 4 (SURVEY.md 6)
    if not cfg["nnet"]:
        return max(64, 16 * cores)
    return max(cores, 8) if cfg["width"] <= 1024 else cores


def run_reference_arm(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n_utts = reference_sample_size(cfg, cores)
    times = []
    frames = 0
    for i in range(args.warmup + args.steps):
        sec, frames, _ = time_reference(cfg, cores, n_utts, 1)
        if i >= args.warmup:
            times.append(sec)
    total = float(sum(times))
    value = frames * len(times) / total
    sample = "%d synthetic 10 s utterances (%d frames) per step, %d host threads, oracle/_ref" % (
        n_utts, frames, cores)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * total / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg["name"], "sample": sample},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": cores, "kind": "reference",
                         "sample": sample},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "rtfx": value / 100.0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- GPU arm
def precision_id(name):
    import pocketkaldi_b200 as pk
    table = {"bf16": pk.PREC_BF16, "bf16x3": pk.PREC_BF16X3, "fp16": pk.PREC_FP16}
    for k, attr in (("fp16x3", "PREC_FP16X3"), ("fp16c8", "PREC_FP16C8"), ("fp16r", "PREC_FP16R")):
        if hasattr(pk, attr):
            table[k] = getattr(pk, attr)
    return table[name]


def uniform_prior(cfg):
    return np.full(cfg["pdfs"], 1.0 / cfg["pdfs"], np.float32)


class Env:
    """What every measurement leg shares: ranks, the library context, peaks."""

    def __init__(self, args):
        import pocketkaldi_b200 as pk
        self.args = args
        self.rank, self.world, self.local, self.dist = dist_setup(args.gpus)
        self.peaks = load_peaks()
        self.ctx = pk.Context(self.local)
        from pocketkaldi_b200.synth import synth_global_cmvn
        self.g = synth_global_cmvn()

    def close(self):
        self.ctx.close()
        if self.dist is not None:
            self.dist.destroy_process_group()


def dump_batch_outputs(batch, cfg, out_dir):
    """Writes what one pass hands its caller: the log-likelihoods (the CMVN features for a config
    without a net), every row when they fit in DUMP_LIMIT, otherwise a fixed seeded sample of
    rows, in ascending row order, next to the row indices."""
    import pocketkaldi_b200 as pk
    which, name, cols = (pk.BUF_LOGLIK, "loglik", cfg["pdfs"]) if cfg["nnet"] else (pk.BUF_FEATS, "feats", 40)
    n = batch.total_frames
    k = min(n, (DUMP_LIMIT - 4096) // (4 * cols + 8))  # 4096: room for the two .npy headers
    rows = np.sort(np.random.default_rng(0).choice(n, k, replace=False)) if k < n else np.arange(n)
    out = np.empty((k, cols), np.float32)
    # one copy per run of consecutive rows
    for run in np.split(np.arange(k), np.flatnonzero(np.diff(rows) != 1) + 1):
        if run.size:
            batch.get_rows_async(which, int(rows[run[0]]), run.size, out[run[0]:])
    batch.ctx.sync()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), out)
    np.save(os.path.join(out_dir, name + "_rows.npy"), rows.astype(np.float64))


def measure_batch(env, cfg, precision, n_utts, steps, warmup, sample_clocks, dump_dir=None):
    """Device-resident throughput of one config: W warm-up passes, K timed passes bracketed by a
    barrier + synchronize, CUDA events on the library's stream, max over ranks. Returns the
    result dict plus the live (am, batch) for the legs that follow (parity, e2e). With dump_dir,
    rank 0 writes the output of the last timed pass there (dump_batch_outputs)."""
    import pocketkaldi_b200 as pk
    from pocketkaldi_b200 import sharding
    args, ctx, rank, local, dist, peaks = env.args, env.ctx, env.rank, env.local, env.dist, env.peaks
    am = None
    if cfg["nnet"]:
        am = pk.AcousticModel(ctx, precision_id(precision)).from_layers(make_layers(cfg), uniform_prior(cfg), 5, 5)
        if precision == "fp16r":
            am.set_refine_margin(REFINE_MARGIN)
    # the nnet reads the 16-bit operand planes the CMVN kernel writes; the FP32 copy of the
    # features is not part of the path to the log-likelihoods (PKB_STAGE_NO_FEATS)
    stages = (pk.STAGE_ALL | pk.STAGE_NO_FEATS) if cfg["nnet"] else (pk.STAGE_FBANK | pk.STAGE_CMVN)
    batch = pk.Batch(ctx, [SAMPLES_10S] * n_utts, env.g, am, prob_scale=0.1)
    batch.synth_pcm(1234, int(sharding.weak_scaling_ids(rank, n_utts)[0]))
    ctx.sync()
    frames = batch.total_frames
    for _ in range(warmup):
        batch.run(stages)
    ctx.sync()
    ctx.profile_enable(True)
    ctx.profile_reset()
    barrier(dist, local)
    sampler = ClockSampler(local) if (rank == 0 and sample_clocks) else None
    ctx.timer_start()
    for _ in range(steps):
        batch.run(stages)
    ms = ctx.timer_stop()
    barrier(dist, local)
    clocks = sampler.stop() if sampler else None
    prof = ctx.profile_get()
    ctx.profile_enable(False)
    ms_max, total_frames = reduce_timing(dist, local, ms, frames)
    value = total_frames * steps / (ms_max * 1e-3)
    if dump_dir is not None and rank == 0:
        dump_batch_outputs(batch, cfg, dump_dir)
    checksum = batch.checksum(pk.BUF_LOGLIK if cfg["nnet"] else pk.BUF_FEATS)

    gemm_launches = prof["gemm"][0] + prof["gemm_final"][0]
    gemm_ms = prof["gemm"][1] + prof["gemm_final"][1]
    refine = None
    if cfg["nnet"] and precision == "fp16r":
        # the selection, gather and scatter kernels of the second pass belong to the nnet's time
        gemm_ms += prof["misc"][1]
        rows, refined = batch.refine_stats()
        refine = {"margin": REFINE_MARGIN, "gemm_rows": rows, "frames_recomputed": refined,
                  "fraction_of_frames": refined / max(frames, 1),
                  "select_gather_scatter_ms_per_step": prof["misc"][1] / steps,
                  "how": "pass 1: one FP16 MMA per product for every frame; pass 2: FP16C8 operands for the "
                         "frames whose two best pdfs are closer than the margin (include/pkb200.h)"}
    fb_ms = prof["fbank"][1] + prof["cmvn"][1]
    front_gbs = 480.0 * frames * steps / (fb_ms * 1e-3) / 1e9 if fb_ms > 0 else None
    cmvn_gbs = 320.0 * frames * steps / (prof["cmvn"][1] * 1e-3) / 1e9 if prof["cmvn"][1] > 0 else None
    fbank_tflops = 16e3 * frames * steps / (prof["fbank"][1] * 1e-3) / 1e12 if prof["fbank"][1] > 0 else None
    if cfg["nnet"]:
        achieved = flops_per_frame(cfg) * frames * steps / (gemm_ms * 1e-3) / 1e12
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "r2_gemm_traffic.json")
        if os.path.exists(tpath):
            t = json.load(open(tpath))
            key = "config%s_%s" % (cfg["key"], precision)
            if key in t:
                # per launch, like `achieved` (FP16R: 2 x (hidden + 1) launches per step)
                traffic = t[key]["dram_bytes_per_frame"] * frames / max(gemm_launches / max(steps, 1), 1)
                traffic_src = "static: %s of profiles/r2_gemm_traffic.json (ncu --set full, " \
                              "dram__bytes_read+write summed over the GEMM launches of one step, " \
                              "scaled by frames; not measured in this run)" % key
        roofline = {"bound": "tensor", "achieved": achieved, "peak": peaks["tensor_sustained"],
                    "unit": "TFLOP/s", "frac": achieved / peaks["tensor_sustained"], "traffic": traffic,
                    "traffic_source": traffic_src,
                    "algorithmic_bytes_per_frame": 160 + 4 * cfg["pdfs"],
                    "algorithmic_flops_per_frame": flops_per_frame(cfg),
                    "hidden_layers_tflops": (flops_per_frame(cfg) - 2 * cfg["width"] * cfg["pdfs"]) * frames
                                            * steps / (prof["gemm"][1] * 1e-3) / 1e12,
                    "output_layer_tflops": 2 * cfg["width"] * cfg["pdfs"] * frames * steps
                                           / (prof["gemm_final"][1] * 1e-3) / 1e12,
                    "kernel": "gemm_kernel (tcgen05, all %d layers%s)" % (
                        cfg["hidden"] + 1, "; both passes plus selection / gather / scatter" if refine else ""),
                    "peak_source": "%s bf16_tflops_sustained (kernel timed inside a long step); only the "
                                   "reference's FLOPs count, the extra MMAs of a split mode do not"
                                   % peaks["src"],
                    "avg_launch_ms": gemm_ms / max(gemm_launches, 1)}
    else:
        roofline = {"bound": "hbm", "achieved": front_gbs, "peak": peaks["hbm"], "unit": "GB/s",
                    "frac": front_gbs / peaks["hbm"], "traffic": None,
                    "kernel": "fbank_kernel + cmvn_kernel (480 algorithmic B/frame)",
                    "peak_source": "%s hbm_gbs" % peaks["src"],
                    "avg_launch_ms": fb_ms / max(prof["fbank"][0] + prof["cmvn"][0], 1)}
    res = {
        "value": value, "unit": "frames/s", "ms_per_step": ms_max / steps, "steps": steps,
        "warmup": warmup, "rtfx": value / 100.0, "dtype": precision if cfg["nnet"] else "f32",
        "config": {"workload": cfg["name"], "utts_per_gpu": n_utts, "frames_per_gpu": frames,
                   "l2": "inputs larger than L2 (PCM %.2f GB%s)" % (
                       batch.total_samples * 2 / 1e9,
                       ", activations > 1 GB per layer" if cfg["nnet"] else ""),
                   "parallelism": "utterance shards, no collective"},
        "roofline": roofline,
        "roofline_frontend": {"bound": "hbm (nominal; the fused fbank kernel is FP32/issue bound)",
                              "achieved": front_gbs, "peak": peaks["hbm"], "unit": "GB/s",
                              "frac": (front_gbs / peaks["hbm"]) if front_gbs else None,
                              "fbank_ms_per_step": prof["fbank"][1] / steps,
                              "cmvn_ms_per_step": prof["cmvn"][1] / steps,
                              # the stand-alone CMVN kernel is the HBM-bound one (SURVEY 8d: 320 B/frame)
                              "cmvn_gbs": cmvn_gbs,
                              "cmvn_frac": (cmvn_gbs / peaks["hbm"]) if cmvn_gbs else None,
                              # SURVEY 8d: ~16 kFLOP/frame against the 74.4 TFLOP/s FP32 FMA peak
                              "fbank_fp32_tflops": fbank_tflops,
                              "fbank_fp32_frac": (fbank_tflops / 74.4) if fbank_tflops else None},
        "kernel_ms_per_step": {k: v[1] / steps for k, v in prof.items()},
        "gpu_launches": int(sum(v[0] for v in prof.values())),
        "clocks": clocks, "checksum": checksum,
    }
    if refine:
        res["refine"] = refine
    return res, am, batch


def parity_ok(par, nnet):
    if par is None:
        return None
    ok = par["fbank_max_rel_err"] <= FEAT_TOL and par["cmvn_max_err_rel_to_max1"] <= FEAT_TOL
    if nnet:
        ok = ok and par["loglik_max_abs_err_unscaled"] <= LL_TOL and par["argmax_agreement"] >= ARGMAX_MIN
    return bool(ok)


def run_gpu_arm(args, cfg):
    import pocketkaldi_b200 as pk
    env = Env(args)
    rank, world = env.rank, env.world
    n_utts = args.utts or cfg["utts"]
    main, am, batch = measure_batch(env, cfg, args.precision, n_utts, args.steps, args.warmup, True,
                                    dump_dir=args.dump_outputs)

    # ---- end to end through the host-buffer API: pinned PCM in, log-likelihoods out, per chunk
    e2e = None if args.no_e2e else run_e2e(env, cfg, am, n_utts, batch)
    if e2e is not None:
        try:
            ceil = d2h_ceiling(env)
            e2e["d2h_ceiling"] = ceil
            e2e["d2h_frac_of_ceiling"] = e2e["d2h_gbs_per_gpu"] / ceil["per_gpu_gbs"]
        except Exception as ex:  # torch is plumbing here; the measurement is optional
            e2e["d2h_ceiling"] = {"unavailable": str(ex)}
    e2e_decode = None
    if cfg["nnet"] and not args.no_e2e:
        e2e_decode = run_e2e_decode(env, cfg, n_utts)

    # ---- parity sample (rank 0) and CPU baseline (rank 0, N=1 only)
    cpu = parity = other_modes = None
    if rank == 0 and not args.no_cpu:
        cores = os.cpu_count() or 1
        try:
            ref_pack = reference_outputs(cfg, env.g, 3)
            batch.run(pk.STAGE_ALL)  # once with the FP32 feature copy for the comparison
            parity = parity_sample(cfg, batch, ref_pack)
            if world == 1:
                n_ref = reference_sample_size(cfg, cores)
                sec, f_ref, _ = time_reference(cfg, cores, n_ref, 1)
                sec1, f1, _ = time_reference(cfg, 1, 1 if cfg["nnet"] else 8, 1)
                cpu = {"value": f_ref / sec, "unit": "frames/s", "cores": cores, "kind": "reference",
                       "sample": "%d synthetic 10 s utterances (%d frames), std::thread pool, oracle/_ref -O2"
                                 % (n_ref, f_ref),
                       "single_thread_value": f1 / sec1}
                if cfg["nnet"] and not args.no_modes:
                    batch.close()  # free HBM before the secondary modes allocate
                    am.close()
                    batch = am = None
                    other_modes = measure_other_modes(env, cfg, ref_pack, args.precision)
        except Exception as e:  # the reference library is test infrastructure; report, don't die
            cpu = {"value": None, "unit": "frames/s", "cores": cores, "kind": "reference",
                   "sample": "unavailable: %s" % e}
    if batch is not None:
        batch.close()
    if am is not None:
        am.close()

    # ---- the other BASELINE configs as sub-objects of the default line (short runs)
    sub = {}
    if args.config == "3" and not args.no_sub:
        barrier(env.dist, env.local)
        sub["config2"] = sub_config(env, "2", args.precision, with_parity=(rank == 0 and not args.no_cpu))
        sub["config4"] = sub_config(env, "4", args.precision, with_parity=(rank == 0 and not args.no_cpu),
                                    n_utts=args.sub_utts4)
        sub["config5"] = measure_stream(env, CONFIGS["5"], args.precision, steps=200, warmup=20)

    if rank == 0:
        line = {
            "metric": METRIC, "value": main["value"], "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": main["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": args.precision if cfg["nnet"] else "f32", "data": "synthetic",
            "config": dict(main["config"], precision=args.precision),
            "rtfx": main["rtfx"],
            "roofline": main["roofline"],
            "roofline_frontend": main["roofline_frontend"],
            "kernel_ms_per_step": main["kernel_ms_per_step"],
            "refine": main.get("refine"),
            "cpu_baseline": cpu,
            "e2e": e2e,
            "e2e_decode": e2e_decode,
            "gpu_launches": main["gpu_launches"],
            "clocks": main["clocks"],
            "checksum": main["checksum"],
            "parity": parity,
            "parity_ok": parity_ok(parity, cfg["nnet"]),
            "precision_modes": other_modes,
            "device": env.ctx.device_name,
        }
        line.update(sub)
        print(json.dumps(line), flush=True)
    env.close()


def sub_config(env, key, precision, with_parity, n_utts=None):
    """One of the other BASELINE configs, measured with the same rules (W >= 3 warm-up passes,
    barrier + synchronize, CUDA events, max over ranks) on a shorter run."""
    import pocketkaldi_b200 as pk
    cfg = CONFIGS[key]
    res, am, batch = measure_batch(env, cfg, precision, n_utts or cfg["utts"], 3, 3, False)
    res.pop("clocks")
    if with_parity:
        try:
            ref_pack = reference_outputs(cfg, env.g, 3 if cfg["nnet"] else 1)
            batch.run(pk.STAGE_ALL)
            res["parity"] = parity_sample(cfg, batch, ref_pack)
            res["parity_ok"] = parity_ok(res["parity"], cfg["nnet"])
        except Exception as e:
            res["parity"] = {"unavailable": str(e)}
    batch.close()
    if am is not None:
        am.close()
    barrier(env.dist, env.local)
    return res


def run_e2e(env, cfg, am, n_utts, main_batch=None):
    """PCM in pinned host memory -> H2D -> hot path -> D2H of the result into pinned host
    memory, chunk by chunk through the batch API, all inside the timed region. Two contexts
    (two CUDA streams, each with its own model copy and chunk batch) alternate so that the
    D2H copy of chunk i overlaps the H2D + kernels of chunk i+1. With a model the result leaves
    the GPU in the compact form (pkb_batch_set_compact: half bits + one FP32 offset per frame,
    finished per look-up by pk_decodable_loglikelihood / pkb_loglik16_expand); --e2e-fp32 moves
    the FP32 matrix instead."""
    import pocketkaldi_b200 as pk
    from pocketkaldi_b200.binding import PinnedArray
    from pocketkaldi_b200.synth import synth_pcm
    args, ctx, rank, local, dist = env.args, env.ctx, env.rank, env.local, env.dist
    chunk = min(args.e2e_chunk, n_utts)
    n_chunks = max(n_utts // chunk, 1)  # whole chunks only; the metric is a rate
    stages = (pk.STAGE_ALL | pk.STAGE_NO_FEATS) if cfg["nnet"] else (pk.STAGE_FBANK | pk.STAGE_CMVN)
    compact = cfg["nnet"] and not args.e2e_fp32
    out_cols = cfg["pdfs"] if cfg["nnet"] else 40
    lanes = []
    for i in range(2):
        c = ctx if i == 0 else pk.Context(local)
        a = am
        if cfg["nnet"] and i == 1:
            a = pk.AcousticModel(c, precision_id(args.precision)).from_layers(
                make_layers(cfg), uniform_prior(cfg), 5, 5)
        cb = pk.Batch(c, [SAMPLES_10S] * chunk, env.g, a, prob_scale=0.1)
        if compact:
            cb.set_compact(True)
        pin_in = PinnedArray((chunk * SAMPLES_10S,), np.int16)
        pin_out = PinnedArray((cb.total_frames, out_cols), np.uint16 if compact else np.float32)
        pin_off = PinnedArray((cb.total_frames,), np.float32) if compact else None
        pin_in.array[:] = synth_pcm(1234, np.arange(chunk) + rank * n_utts + i * chunk,
                                    SAMPLES_10S).reshape(-1)
        lanes.append((c, a, cb, pin_in, pin_out, pin_off))
    h2d = lanes[0][3].array.nbytes * n_chunks
    d2h = (lanes[0][4].array.nbytes + (lanes[0][5].array.nbytes if compact else 0)) * n_chunks

    def step():
        for k in range(n_chunks):
            c, a, cb, pin_in, pin_out, pin_off = lanes[k & 1]
            c.sync()  # this lane's previous chunk has fully landed in its pinned buffer
            cb.set_pcm(pin_in.array)
            cb.run(stages)
            if compact:
                cb.get_rows_async(pk.BUF_LOGLIK16, 0, cb.total_frames, pin_out.array)
                cb.get_rows_async(pk.BUF_LOGLIK_OFF, 0, cb.total_frames, pin_off.array)
            else:
                cb.get_rows_async(pk.BUF_LOGLIK if cfg["nnet"] else pk.BUF_FEATS, 0, cb.total_frames,
                                  pin_out.array)
        for lane in lanes:
            lane[0].sync()

    for _ in range(min(args.warmup, 2)):
        step()
    barrier(dist, local)
    steps = max(1, min(args.steps, args.e2e_steps))
    t0 = time.perf_counter()
    ctx.timer_start()
    for _ in range(steps):
        step()
    ms = ctx.timer_stop()
    wall_ms = (time.perf_counter() - t0) * 1e3
    ms = max(ms, wall_ms)  # two streams: the host wall clock covers both lanes
    barrier(dist, local)
    ms_max, frames = reduce_timing(dist, local, ms, lanes[0][2].total_frames * n_chunks)
    check = None
    if compact:
        fin = bool(np.isfinite(lanes[0][5].array).all() and np.isfinite(lanes[1][5].array).all())
        if main_batch is not None:
            # lane 0 holds the first utterances of the main batch: the expanded compact rows must
            # agree with the FP32 rows of the device-resident run (unscaled bar: 2e-2)
            n = FRAMES_10S
            want = np.empty((n, out_cols), np.float32)
            main_batch.get_rows_async(pk.BUF_LOGLIK, 0, n, want)
            ctx.sync()
            got = lanes[0][2].expand_compact(lanes[0][4].array[:n], lanes[0][5].array[:n], 0.1)
            check = {"frames": n, "max_abs_err_unscaled_vs_fp32_output": float(np.max(np.abs(got - want)) / 0.1),
                     "argmax_agreement_vs_fp32_output": float(np.mean(got.argmax(1) == want.argmax(1)))}
    else:
        fin = bool(np.isfinite(lanes[0][4].array[::997]).all() and np.isfinite(lanes[1][4].array[::997]).all())
    for i, (c, a, cb, pin_in, pin_out, pin_off) in enumerate(lanes):
        cb.close()
        pin_in.free()
        pin_out.free()
        if pin_off is not None:
            pin_off.free()
        if i == 1:
            if cfg["nnet"]:
                a.close()
            c.close()
    return {"value": frames * steps / (ms_max * 1e-3), "unit": "frames/s",
            "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "steps": steps,
            "ms_per_step": ms_max / steps, "chunk_utts": chunk, "chunks_per_step": n_chunks,
            "d2h_gbs_per_gpu": d2h * steps / (ms_max * 1e-3) / 1e9,
            "result_form": ("compact: fp16(loglik/prob_scale - off[frame]) + FP32 off[frame], %d B/frame; the "
                            "consumer finishes prob_scale*(half+off) per look-up" % (2 * out_cols + 4))
                           if compact else "FP32 matrix, %d B/frame" % (4 * out_cols),
            "compact_check": check,
            "finite": fin, "timing": "host wall clock over both streams (>= the CUDA-event time of stream 0)",
            "api": "2 x (pkb_batch_set_pcm_i16 + pkb_batch_run + pkb_batch_get_rows), pinned host "
                   "buffers, two contexts alternating so D2H overlaps the next chunk"}


def d2h_ceiling(env, gib=1, reps=3):
    """What this box gives N ranks copying device -> pinned host memory at the same time (plain
    cudaMemcpyAsync of 1 GiB per rank, no kernels): the ceiling of the e2e leg, whose result bytes
    cross the same links. Aggregate = bytes of all ranks / max-over-ranks time."""
    import torch
    dev = torch.device("cuda", env.local)
    n = gib << 30
    src = torch.empty(n, dtype=torch.uint8, device=dev)
    dst = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize(dev)
    barrier(env.dist, env.local)
    t0 = time.perf_counter()
    for _ in range(reps):
        dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize(dev)
    ms = (time.perf_counter() - t0) * 1e3
    barrier(env.dist, env.local)
    ms_max, total = reduce_timing(env.dist, env.local, ms, float(n) * reps)
    del src, dst
    torch.cuda.empty_cache()
    return {"aggregate_gbs": total / (ms_max * 1e-3) / 1e9, "per_gpu_gbs": total / env.world / (ms_max * 1e-3) / 1e9,
            "how": "%d rank(s) x %d x %d GiB cudaMemcpyAsync device -> pinned host at the same time" % (env.world, reps, gib)}


def run_e2e_decode(env, cfg, n_utts):
    """PCM in pinned host memory -> H2D -> fbank/CMVN/nnet -> GPU Viterbi (pkb_batch_decode) -> word
    ids on the host: the path on which the [frames x pdfs] matrix never crosses PCIe (SURVEY 8(f)-4).
    Graph: the 40-word loop of tools/decode_demo.py over the config's pdfs; beam 16 like the
    reference decoder. One context, chunk after chunk (the decode call synchronises)."""
    import pocketkaldi_b200 as pk
    from pocketkaldi_b200.binding import PinnedArray
    from pocketkaldi_b200.synth import synth_pcm
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from decode_demo import word_loop_graph
    args, ctx, rank, local, dist = env.args, env.ctx, env.rank, env.local, env.dist
    chunk = min(4 * args.e2e_chunk, n_utts)   # one thread block per utterance: fill the machine
    n_chunks = max(n_utts // chunk, 1)
    graph, tid2pdf = word_loop_graph(40, 3, cfg["pdfs"])
    am = pk.AcousticModel(ctx, precision_id(args.precision)).from_layers(
        make_layers(cfg), uniform_prior(cfg), 5, 5, tid2pdf=np.asarray(tid2pdf, np.int32))
    fst = pk.Fst(ctx, graph=graph)
    cb = pk.Batch(ctx, [SAMPLES_10S] * chunk, env.g, am, prob_scale=0.1)
    pin_in = PinnedArray((chunk * SAMPLES_10S,), np.int16)
    pin_in.array[:] = synth_pcm(1234, np.arange(chunk) + rank * n_utts, SAMPLES_10S).reshape(-1)
    stages = pk.STAGE_ALL | pk.STAGE_NO_FEATS
    words = 0

    def step():
        nonlocal words
        for _ in range(n_chunks):
            cb.set_pcm(pin_in.array)
            cb.run(stages)
            hyps, _ = cb.decode(fst)
            words = sum(len(h) for h in hyps if h is not None)
            if any(h is None for h in hyps):
                raise RuntimeError("GPU Viterbi ran out of token capacity")

    step()
    barrier(dist, local)
    steps = max(1, min(args.steps, args.e2e_steps))
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    ms = (time.perf_counter() - t0) * 1e3
    barrier(dist, local)
    ms_max, frames = reduce_timing(dist, local, ms, cb.total_frames * n_chunks)
    res = {"value": frames * steps / (ms_max * 1e-3), "unit": "frames/s", "steps": steps,
           "ms_per_step": ms_max / steps, "chunk_utts": chunk, "chunks_per_step": n_chunks,
           "h2d_bytes_per_step": int(pin_in.array.nbytes * n_chunks),
           "d2h_bytes_per_step": int(chunk * (256 + 2) * 4 * n_chunks),
           "words_per_chunk": int(words),
           "graph": "40-word loop, 121 states, 1800 arcs, beam 16 (tools/decode_demo.py)",
           "api": "pkb_batch_set_pcm_i16 + pkb_batch_run + pkb_batch_decode (word ids out), host wall clock"}
    cb.close()
    fst.close()
    am.close()
    pin_in.free()
    return res


def reference_outputs(cfg, g, n_utts=1):
    """The unmodified reference on the first utterances of the synthetic corpus (checker only)."""
    from oracle.oracle import Reference
    from pocketkaldi_b200.synth import synth_pcm
    ref = Reference()
    raws, feats, lls = [], [], []
    tmp = am = None
    if cfg["nnet"]:
        tmp = tempfile.TemporaryDirectory(prefix="pkb_parity_")
        conf, _, _ = write_reference_model(cfg, tmp.name)
        am = ref.am_load(conf)
    for u in range(n_utts):
        pcm = synth_pcm(1234, [u], SAMPLES_10S)[0].astype(np.float32)
        raws.append(ref.fbank(pcm))
        feats.append(ref.cmvn(raws[-1], g))
        if am:
            lls.append(ref.am_compute(am, feats[-1]) * np.float32(0.1))
    if am:
        ref.am_free(am)
        tmp.cleanup()
    return np.concatenate(raws), np.concatenate(feats), (np.concatenate(lls) if lls else None)


def parity_sample(cfg, batch, ref_pack):
    """GPU output of the first utterances of the batch against reference_outputs()."""
    import pocketkaldi_b200 as pk
    raw, feats, ll_ref = ref_pack
    n = int(raw.shape[0])
    out = {"frames": n}
    got_raw = np.empty((n, 40), np.float32)
    batch.get_rows_async(pk.BUF_RAW, 0, n, got_raw)
    got_ft = np.empty((n, 40), np.float32)
    batch.get_rows_async(pk.BUF_FEATS, 0, n, got_ft)
    batch.ctx.sync()
    out["fbank_max_rel_err"] = float(np.max(np.abs(got_raw - raw) / np.abs(raw)))
    out["cmvn_max_err_rel_to_max1"] = float(np.max(np.abs(got_ft - feats) / np.maximum(1.0, np.abs(feats))))
    if ll_ref is not None:
        got = np.empty((n, cfg["pdfs"]), np.float32)
        batch.get_rows_async(pk.BUF_LOGLIK, 0, n, got)
        batch.ctx.sync()
        out["loglik_max_abs_err_unscaled"] = float(np.max(np.abs(got - ll_ref)) / 0.1)
        agree = got.argmax(1) == ll_ref.argmax(1)
        out["argmax_agreement"] = float(np.mean(agree))
        out["argmax_flips"] = int(np.sum(~agree))
        top2 = np.sort(ll_ref, axis=1)[:, -2:] / 0.1
        clear = (top2[:, 1] - top2[:, 0]) > 2e-2   # frames whose reference margin exceeds the LL bar
        out["argmax_agreement_margin_gt_2e-2"] = float(np.mean(agree[clear])) if clear.any() else None
        out["frames_with_margin_gt_2e-2"] = float(np.mean(clear))
        out["tolerance"] = "north_star: |dLL| <= 2e-2, argmax agreement >= 0.999"
    return out


def measure_other_modes(env, cfg, ref_pack, skip):
    """Throughput + parity of the other GEMM precisions on a 512-utterance batch (same net)."""
    import pocketkaldi_b200 as pk
    ctx = env.ctx
    names = ["bf16", "fp16", "bf16x3"] + [k for k, a in (("fp16x3", "PREC_FP16X3"), ("fp16c8", "PREC_FP16C8"),
                                                          ("fp16r", "PREC_FP16R")) if hasattr(pk, a)]
    out = {}
    layers = make_layers(cfg)
    prior = uniform_prior(cfg)
    for name in names:
        if name == skip:
            continue
        am = pk.AcousticModel(ctx, precision_id(name)).from_layers(layers, prior, 5, 5)
        b = pk.Batch(ctx, [SAMPLES_10S] * 512, env.g, am, prob_scale=0.1)
        b.synth_pcm(1234, 0)
        for _ in range(3):
            b.run(pk.STAGE_ALL)
        ctx.sync()
        ctx.timer_start()
        for _ in range(3):
            b.run(pk.STAGE_ALL)
        ms = ctx.timer_stop()
        par = parity_sample(cfg, b, ref_pack)
        out[name] = {"value": b.total_frames * 3 / (ms * 1e-3), "unit": "frames/s",
                     "utts": 512, "parity": par, "parity_ok": parity_ok(par, True)}
        b.close()
        am.close()
    return out


def measure_stream(env, cfg, precision, steps, warmup, dump_dir=None):
    """BASELINE config 5: chunk latency from "chunk in pinned host memory" to "log-likelihoods in
    pinned host memory" (host wall clock around the synchronous pkb_stream_push_i16). With
    dump_dir, rank 0 writes the log-likelihoods of the last timed push there."""
    import pocketkaldi_b200 as pk
    from pocketkaldi_b200.binding import PinnedArray
    from pocketkaldi_b200.synth import synth_pcm
    args, ctx, rank, local, dist = env.args, env.ctx, env.rank, env.local, env.dist
    S, chunk = cfg["utts"], 2560
    am = pk.AcousticModel(ctx, precision_id(precision)).from_layers(make_layers(cfg), uniform_prior(cfg), 5, 5)
    st = pk.Stream(ctx, am, S, chunk, env.g, 0.1)
    n_chunks = warmup + steps
    pin_in = PinnedArray((S, chunk), np.int16)
    pin_out = PinnedArray((S, st.max_frames, cfg["pdfs"]), np.float32)
    audio = synth_pcm(1234, np.arange(S) + rank * S, chunk * 8)
    lat, frames = [], 0
    ctx.profile_reset()
    barrier(dist, local)
    t_all0 = None
    for k in range(n_chunks):
        pin_in.array[:] = audio[:, (k % 8) * chunk:((k % 8) + 1) * chunk]
        if k == warmup:
            ctx.profile_reset()
            t_all0 = time.perf_counter()
        t0 = time.perf_counter()
        o = st.push(pin_in.array, out=pin_out.array)
        t1 = time.perf_counter()
        if k >= warmup:
            lat.append((t1 - t0) * 1e3)
            frames += o.shape[1] * S
    total_ms = (time.perf_counter() - t_all0) * 1e3
    barrier(dist, local)
    prof = ctx.profile_get()
    ms_max, frames_all = reduce_timing(dist, local, total_ms, frames)
    if dump_dir is not None and rank == 0:
        os.makedirs(dump_dir, exist_ok=True)
        np.save(os.path.join(dump_dir, "loglik.npy"), np.ascontiguousarray(o))
    lat = np.array(lat)
    # the same with the compact output form (half the D2H bytes, finished per look-up by the consumer)
    st.flush(out=pin_out.array)
    st.set_compact(True)
    pin_h = PinnedArray((S, st.max_frames, cfg["pdfs"]), np.uint16)
    pin_o = PinnedArray((S, st.max_frames), np.float32)
    lat_c = []
    for k in range(n_chunks):
        pin_in.array[:] = audio[:, (k % 8) * chunk:((k % 8) + 1) * chunk]
        t0 = time.perf_counter()
        st.push_compact(pin_in.array, pin_h.array, pin_o.array)
        t1 = time.perf_counter()
        if k >= warmup:
            lat_c.append((t1 - t0) * 1e3)
    lat_c = np.array(lat_c)
    value = frames_all / (ms_max * 1e-3)
    res = {
        "value": value, "unit": "frames/s", "steps": steps, "warmup": warmup,
        "ms_per_step": ms_max / steps, "dtype": precision, "rtfx": value / 100.0,
        "config": {"workload": cfg["name"], "streams_per_gpu": S, "chunk_samples": chunk,
                   "timing": "host wall clock around the synchronous push (H2D + kernels + D2H), rank 0"},
        "latency_ms": {"p50": float(np.percentile(lat, 50)), "p99": float(np.percentile(lat, 99)),
                       "mean": float(lat.mean()), "max": float(lat.max())},
        "latency_ms_compact_output": {"p50": float(np.percentile(lat_c, 50)), "p99": float(np.percentile(lat_c, 99)),
                                      "mean": float(lat_c.mean()), "max": float(lat_c.max()),
                                      "d2h_bytes_per_step": int(S * (chunk // 160) * (cfg["pdfs"] * 2 + 4))},
        "launch_path": "CUDA graph replay of the steady-state push (PKB_STREAM_GRAPH=0 disables it)",
        "e2e": {"value": value, "unit": "frames/s",
                "h2d_bytes_per_step": int(pin_in.array.nbytes),
                "d2h_bytes_per_step": int(S * (chunk // 160) * cfg["pdfs"] * 4)},
        "gpu_launches": int(sum(v[0] for v in prof.values())),
    }
    st.close()
    am.close()
    pin_in.free()
    pin_out.free()
    pin_h.free()
    pin_o.free()
    return res


def run_stream_arm(args, cfg):
    env = Env(args)
    sampler = ClockSampler(env.local) if env.rank == 0 else None
    res = measure_stream(env, cfg, args.precision, args.steps, args.warmup, dump_dir=args.dump_outputs)
    clocks = sampler.stop() if sampler else None
    if env.rank == 0:
        line = {"metric": METRIC, "n_gpus": env.world, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "data": "synthetic", "clocks": clocks, "device": env.ctx.device_name}
        line.update(res)
        print(json.dumps(line), flush=True)
    env.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="3", choices=sorted(CONFIGS))
    ap.add_argument("--precision", default=DEFAULT_PRECISION,
                    choices=["bf16", "bf16x3", "fp16", "fp16x3", "fp16c8", "fp16r"])
    ap.add_argument("--utts", type=int, default=0, help="utterances per GPU (default: the config's)")
    ap.add_argument("--e2e-chunk", type=int, default=256)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer leg (profiling runs)")
    ap.add_argument("--e2e-fp32", action="store_true", help="e2e leg moves the FP32 matrix instead of the compact rows")
    ap.add_argument("--no-sub", action="store_true", help="skip the config 2/4/5 sub-objects")
    ap.add_argument("--no-modes", action="store_true", help="skip the other precision modes")
    ap.add_argument("--sub-utts4", type=int, default=512, help="utterances per GPU of the config-4 sub-run")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the output of the last timed step as DIR/<name>.npy (float32, row "
                         "indices in float64; at most 64 MB in all, a fixed seeded row sample of "
                         "larger outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; --impl reference has none")
    cfg = CONFIGS[args.config]
    if args.impl == "reference":
        run_reference_arm(args, cfg)
    elif cfg.get("stream"):
        run_stream_arm(args, cfg)
    else:
        run_gpu_arm(args, cfg)


if __name__ == "__main__":
    main()
