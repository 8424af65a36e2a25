"""GPU Viterbi (SURVEY 8(f)-4, pkb_batch_decode) against the reference's own decoder: the
unmodified reference CLI (oracle/_ref/pocketkaldi_ref: CPU nnet + src/decoder.cc), or where it is
not built the host restatement of that path (oracle/decoder.py), must print the same words, and
the same per-frame weight, for every utterance."""

import os
import subprocess

import numpy as np
import pytest

import pocketkaldi_b200 as pk
from oracle.decoder import host_decode
from pocketkaldi_b200 import formats
from pocketkaldi_b200.synth import synth_global_cmvn, synth_pcm

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_CLI = os.path.join(ROOT, "oracle", "_ref", "pocketkaldi_ref")


@pytest.fixture(scope="module")
def ctx():
    c = pk.Context(0)
    yield c
    c.close()


def ref_cli(conf, scp):
    out = subprocess.run([REF_CLI, conf, scp], stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600,
                         check=True).stdout.decode()
    res = []
    for line in out.strip().splitlines():
        _, hyp, llpf = line.split("\t")
        res.append((hyp.strip(), float(llpf)))
    return res


def gpu_decode(ctx, conf, pcms, g, precision=pk.PREC_BF16X3, **kw):
    table = formats.read_conf(conf)
    am = pk.AcousticModel(ctx, precision).Read(conf)
    fst = pk.Fst(ctx, path=formats.conf_path(conf, table["fst"]))
    b = pk.Batch(ctx, [len(p) for p in pcms], g, am, prob_scale=0.1)
    b.set_pcm(np.ascontiguousarray(np.concatenate(pcms), np.int16))
    b.run(pk.STAGE_ALL)
    hyps, wts = b.decode(fst, **kw)
    frames = b.num_frames.copy()
    b.close()
    fst.close()
    am.close()
    return hyps, wts, frames


def coloured(seed, n):
    """int16 noise whose spectral tilt changes every 0.25 s (first-order IIR with a random pole), so
    that the best path walks through several words."""
    rng = np.random.default_rng(seed)
    x = synth_pcm(seed, [0], n)[0].astype(np.float64)
    poles = rng.choice([-0.9, -0.6, 0.0, 0.6, 0.9], size=n // 4000 + 1)
    out = np.empty(n)
    prev = 0.0
    for s in range(0, n, 4000):
        a = poles[s // 4000]
        for i in range(s, min(s + 4000, n)):
            prev = x[i] + a * prev
            out[i] = prev * np.sqrt(1 - a * a)
    return np.clip(np.round(out), -32768, 32767).astype(np.int16)


def words_of(ids, words):
    return " ".join(words[i] for i in ids)


def test_toy_model_words_match_the_reference(ctx, golden, toy_conf):
    gold = {}
    for line in open(os.path.join(ROOT, "tests", "golden", "toy_decode_ref.txt")):
        name, hyp, llpf = line.rstrip("\n").split("\t")
        gold[name] = (hyp.strip(), float(llpf))
    # tests/golden/toy/toy.sym: word ids of the toy graph
    sym = open(os.path.join(os.path.dirname(toy_conf), formats.read_conf(toy_conf)["symbol_table"]), "rb").read()
    n, buflen = np.frombuffer(sym[8:16], "<i4")
    idx = np.frombuffer(sym[16:16 + 4 * n], "<i4")
    buf = sym[16 + 4 * n:]
    words = [buf[i:buf.index(b"\0", i)].decode() for i in idx]
    pcms = [golden["hello_pcm"], golden["cat_pcm"], golden["hello_pcm"]]
    for prec in (pk.PREC_BF16X3, pk.PREC_FP16C8, pk.PREC_FP16R):
        hyps, wts, frames = gpu_decode(ctx, toy_conf, pcms, golden["cmvn_stats"], prec)
        for name, h, w, T in zip(("hello", "cat", "hello"), hyps, wts, frames):
            assert words_of(h, words) == gold[name][0], (name, h)
            assert abs(w / T - gold[name][1]) < 2e-3


def eps_graph(n_words, n_hmm, num_pdfs):
    """Word loop through a hub with epsilon arcs: start -eps-> hub; hub -> word entry (emitting, word
    label); word end -eps-> tail -eps(word-end label)-> hub: closures of depth two, output labels on
    epsilon arcs, and word ends that are final."""
    arcs, tid2pdf = [], [0]
    hub, tail0 = 1, 2
    state_of = lambda w, s: 2 + n_words + w * n_hmm + s
    tid = 1
    enter = {}
    for w in range(n_words):
        for s in range(n_hmm):
            pdf = (w * n_hmm + s) % num_pdfs
            arcs.append((state_of(w, s), state_of(w, s), tid, 0, 0.05))
            tid2pdf.append(pdf)
            tid += 1
            enter[(w, s)] = tid
            tid2pdf.append(pdf)
            tid += 1
    arcs.append((0, hub, 0, 0, 0.1))
    for w in range(n_words):
        arcs.append((hub, state_of(w, 0), enter[(w, 0)], w + 1, 0.2 + 0.01 * w))
        for s in range(1, n_hmm):
            arcs.append((state_of(w, s - 1), state_of(w, s), enter[(w, s)], 0, 0.1))
        arcs.append((state_of(w, n_hmm - 1), tail0 + w, 0, 0, 0.05))          # epsilon, no label
        arcs.append((tail0 + w, hub, 0, n_words + 1, 0.02 * (w + 1)))         # epsilon with a label
    finals = {state_of(w, n_hmm - 1): 0.3 for w in range(n_words)}
    finals[hub] = 0.0
    return (2 + n_words + n_words * n_hmm, 0, finals, arcs), tid2pdf


@pytest.mark.parametrize("kind", ["loop", "eps", "loop_big"])
def test_random_graphs_against_the_reference_cli(ctx, oracle, tmp_path, kind):
    # "loop" / "eps": small graphs, token tables in shared memory; "loop_big": 541 states, the
    # tables live in the global workspace. The reference CLI where oracle/_ref is built, otherwise
    # the host restatement of its path (oracle/decoder.py, pinned by tests/test_oracle.py)
    rng = np.random.default_rng({"loop": 1, "eps": 2, "loop_big": 3}[kind])
    P = 600 if kind == "loop_big" else 96
    layers = formats.make_dnn(rng, 440, 96, 2, P)
    # make the acoustic scores decisive enough that a 1e-4 difference between the CPU and the GPU
    # nnet cannot flip a path, but keep several words alive in the beam
    layers[-2] = ("linear", (layers[-2][1] * 3.0).astype(np.float32), layers[-2][2])
    prior = rng.uniform(0.5, 1.5, P).astype(np.float32)
    prior /= prior.sum()
    if kind.startswith("loop"):
        import tools.decode_demo as demo
        nw = 180 if kind == "loop_big" else 12
        fst, tid2pdf = demo.word_loop_graph(nw, 3, P)
        words = ["<eps>"] + ["w%03d" % i for i in range(nw)]
    else:
        fst, tid2pdf = eps_graph(10, 3, P)
        words = ["<eps>"] + ["w%02d" % i for i in range(10)] + ["</w>"]
    g = synth_global_cmvn()
    conf = formats.write_model_dir(str(tmp_path), kind, layers, prior, 5, 5, tid2pdf, cmvn_stats=g, fst=fst,
                                   words=words)
    # (an utterance shorter than one frame aborts the reference CLI: SURVEY appendix C)
    lens = [16000, 24000, 8000, 32000, 400, 12345, 48000, 20000, 28000]
    pcms = [coloured(100 + u, n) for u, n in enumerate(lens)]
    paths = []
    for u, p in enumerate(pcms):
        paths.append(str(tmp_path / ("u%d.wav" % u)))
        formats.write_wav16(paths[-1], p)
    scp = str(tmp_path / "all.scp")
    open(scp, "w").write("\n".join(paths) + "\n")
    if os.path.exists(REF_CLI):
        ref = ref_cli(conf, scp)
    else:
        ref = [(words_of(ids, words), llpf)
               for ids, llpf in host_decode(oracle, fst, tid2pdf, layers, prior, g, pcms)]
    hyps, wts, frames = gpu_decode(ctx, conf, pcms, g)
    assert len(ref) == len(hyps)
    for u, ((rh, rl), h, w, T) in enumerate(zip(ref, hyps, wts, frames)):
        assert h is not None, u
        assert words_of(h, words) == rh, (u, words_of(h, words), rh)
        assert abs(w / T - rl) < 2e-3, (u, w / T, rl)
    assert any(len(h) > 2 for h in hyps)   # the fixture really exercises multi-word paths


def test_capacity_overflow_is_reported_not_silent(ctx, tmp_path):
    rng = np.random.default_rng(3)
    import tools.decode_demo as demo
    P = 640
    layers = formats.make_dnn(rng, 440, 32, 1, P)
    prior = np.full(P, 1.0 / P, np.float32)
    fst, tid2pdf = demo.word_loop_graph(200, 3, P)   # 601 states: tables in the global workspace
    g = synth_global_cmvn()
    conf = formats.write_model_dir(str(tmp_path), "ovf", layers, prior, 5, 5, tid2pdf, cmvn_stats=g, fst=fst,
                                   words=["<eps>"] + ["w%03d" % i for i in range(200)])
    pcms = [synth_pcm(5, [0], 16000)[0], synth_pcm(5, [1], 16000)[0]]
    hyps, _, _ = gpu_decode(ctx, conf, pcms, g, max_tokens=64)
    assert hyps[0] is None and hyps[1] is None  # hundreds of live states do not fit 64 tokens: flagged
    hyps, _, _ = gpu_decode(ctx, conf, pcms, g, max_tokens=1024)
    assert all(h is not None and len(h) > 0 for h in hyps)   # and the workspace is clean afterwards


def test_tid2pdf_outside_the_model_is_rejected(ctx):
    # the reference would index past the log-likelihood row (src/decodable.cc:24-31); here the
    # decode call reports it
    import tools.decode_demo as demo
    P = 64
    layers = formats.make_dnn(np.random.default_rng(8), 440, 32, 1, P)
    graph, tid2pdf = demo.word_loop_graph(4, 3, P)
    bad = np.asarray(tid2pdf, np.int32).copy()
    bad[-1] = P  # one past the last pdf
    am = pk.AcousticModel(ctx, pk.PREC_BF16X3).from_layers(layers, np.full(P, 1.0 / P, np.float32), 5, 5, tid2pdf=bad)
    fst = pk.Fst(ctx, graph=graph)
    b = pk.Batch(ctx, [16000], synth_global_cmvn(), am, prob_scale=0.1)
    b.synth_pcm(1, 0)
    b.run(pk.STAGE_ALL)
    with pytest.raises(pk.PkbError):
        b.decode(fst)
    b.close()
    fst.close()
    am.close()
