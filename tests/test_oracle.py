"""Pins the CPU restatement (oracle/pk_oracle.c) against the reference's own golden
vectors and known answers, and against the compiled reference (oracle/_ref) when built.
Runs without a GPU."""

import numpy as np
import pytest

from pocketkaldi_b200 import formats
from pocketkaldi_b200.synth import synth_pcm


def rel_err(a, b):
    return np.max(np.abs(a - b) / np.maximum(np.abs(b), 1.0))


# ---------------------------------------------------------------- reference golden vectors
def test_srfft_known_answer(oracle, golden):
    # test/srfft_test.cc:273-289 (reference tolerance 1e-6 abs with its own split-radix
    # ordering; the restatement's radix-2 ordering is held to 2e-6 relative to max(1,|x|))
    y = oracle.srfft(golden["srfft128_in"])
    assert rel_err(y, golden["srfft128_out"]) < 2e-6


def test_num_frames(oracle):
    # src/fbank.cc:35-42
    for n, t in ((0, 0), (399, 0), (400, 1), (559, 1), (560, 2), (160000, 998), (7802, 47)):
        assert oracle.num_frames(n) == t


def test_mel_table_shape(oracle):
    # SURVEY.md 3.3: offsets 1..225, widths 3..31, 492 non-zero weights, bins 0 and 256 unused
    w, off, wid = oracle.mel_table()
    assert off.min() == 1 and off.max() == 225
    assert wid.min() == 3 and wid.max() == 31
    assert int((w != 0).sum()) == 492
    assert np.all(w[:, 0] == 0)


def test_fbank_vs_kaldi_golden(oracle, golden):
    # test/fbank_test.cc:15-56; the golden text has 7 significant digits and the reference
    # itself sits 2.2e-5 from it (SURVEY.md section 4), hence 5e-5 abs.
    fb = oracle.fbank(golden["hello_pcm"].astype(np.float32))
    assert fb.shape == (47, 40)
    assert np.max(np.abs(fb - golden["hello_fbank_kaldi"])) < 5e-5


@pytest.mark.parametrize("name", ["hello", "cat", "noise10", "short400", "short559", "short560"])
def test_fbank_vs_compiled_reference(oracle, golden, name):
    if name + "_pcm" in golden:
        pcm = golden[name + "_pcm"]
    else:
        seed, utt, n = golden[name + "_spec"]
        pcm = synth_pcm(int(seed), [int(utt)], int(n))[0]
    fb = oracle.fbank(pcm.astype(np.float32))
    ref = golden[name + "_fbank_ref"]
    assert fb.shape == ref.shape
    assert np.max(np.abs(fb - ref) / np.abs(ref)) < 1e-5


def test_cmvn_vs_kaldi_golden(oracle, golden):
    # test/cmvn_test.cc:33-82 (one-sided 1e-5 in the reference; it sits 1.2e-5 away itself)
    y = oracle.cmvn(golden["hello_fbank_ref"], golden["cmvn_stats"])
    assert np.max(np.abs(y - golden["hello_cmvn_kaldi"])) < 5e-5


@pytest.mark.parametrize("name", ["hello", "cat", "noise10", "noise12", "short400", "short560"])
def test_cmvn_bit_exact_vs_compiled_reference(oracle, golden, name):
    # Given the reference's raw fbank, the restatement reproduces CMVN::GetFrame exactly,
    # including the float running sum beyond the 600-frame window (noise12: 1248 frames).
    y = oracle.cmvn(golden[name + "_fbank_ref"], golden["cmvn_stats"])
    assert np.array_equal(y, golden[name + "_cmvn_ref"])


def test_nnet_known_answers(oracle, golden):
    # test/nnet_test.cc:23-110, tolerance 1e-6 as in CheckEq
    y = oracle.linear(golden["nnet_kat_x"], golden["nnet_kat_W"], golden["nnet_kat_b"])
    assert np.max(np.abs(y - golden["nnet_kat_linear_y"])) < 1e-6
    x4 = golden["nnet_kat_x4"]
    assert np.max(np.abs(oracle.nnet(x4, [("softmax",)]) - golden["nnet_kat_softmax_y"])) < 1e-6
    assert np.max(np.abs(oracle.nnet(x4, [("relu",)]) - golden["nnet_kat_relu_y"])) < 1e-6
    yn = oracle.nnet(x4, [("normalize",)])
    assert abs(float((yn.astype(np.float64) ** 2).sum()) - 4.0) < 1e-4


@pytest.mark.parametrize("m,n,k", [(512, 512, 512), (100, 100, 1), (1, 1, 1), (121, 233, 17)])
def test_gemm_differential(oracle, m, n, k):
    # test/gemm_test.cc:32-62: packed GEMM vs naive triple loop, max diff < 0.01
    rng = np.random.default_rng(m * 1000 + n)
    A = rng.random((m, k), dtype=np.float32)
    B = rng.random((k, n), dtype=np.float32)
    y = oracle.linear(A, np.ascontiguousarray(B.T), np.zeros(n, np.float32))
    assert np.max(np.abs(y - oracle.simple_matmat(A, B))) < 0.01


def test_splice_edges(oracle):
    # src/am.cc:65-88: clamped indices
    f = np.arange(12, dtype=np.float32).reshape(4, 3)
    s = oracle.splice(f, 2, 1)
    assert s.shape == (4, 12)
    assert np.array_equal(s[0], np.concatenate([f[0], f[0], f[0], f[1]]))
    assert np.array_equal(s[3], np.concatenate([f[1], f[2], f[3], f[3]]))


@pytest.mark.parametrize("name", ["hello", "cat", "noise10"])
def test_am_loglik_vs_compiled_reference(oracle, golden, toy_conf, name):
    conf = formats.read_conf(toy_conf)
    layers = formats.read_nnet(formats.conf_path(toy_conf, conf["nnet"]))
    prior = formats.read_vector(formats.conf_path(toy_conf, conf["prior"]))
    ll = oracle.am_compute(golden[name + "_cmvn_ref"], layers, prior,
                           int(conf["left_context"]), int(conf["right_context"]))
    ref = golden[name + "_toy_loglik_ref"]
    assert ll.shape == ref.shape
    assert np.max(np.abs(ll - ref)) < 2e-5
    assert np.mean(ll.argmax(1) == ref.argmax(1)) == 1.0


def test_decodable_vs_compiled_reference(oracle, golden, toy_conf):
    conf = formats.read_conf(toy_conf)
    layers = formats.read_nnet(formats.conf_path(toy_conf, conf["nnet"]))
    prior = formats.read_vector(formats.conf_path(toy_conf, conf["prior"]))
    tid2pdf = formats.read_vector(formats.conf_path(toy_conf, conf["tid2pdf"]), dtype="<i4")
    lp = oracle.decodable(golden["hello_cmvn_ref"], layers, prior, 5, 5, 0.1)
    tids = np.arange(1, 25)
    got = lp[:, tid2pdf[tids]]
    assert np.max(np.abs(got - golden["hello_toy_decodable_ref"])) < 2e-6
    last = golden["hello_toy_islast_ref"]
    assert last.sum() == 1 and last[-1] == 1


def test_host_decoder_reproduces_the_reference_toy_decodes(oracle, golden, toy_conf):
    # the reference CLI's words and per-frame weight on its two test wavs (tests/golden/make_golden.py)
    import importlib.util
    import os
    from oracle.decoder import host_decode
    here = os.path.dirname(toy_conf)
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(here, "..", "make_golden.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    graph, _, _ = mg.toy_graph()
    conf = formats.read_conf(toy_conf)
    layers = formats.read_nnet(formats.conf_path(toy_conf, conf["nnet"]))
    prior = formats.read_vector(formats.conf_path(toy_conf, conf["prior"]))
    tid2pdf = formats.read_vector(formats.conf_path(toy_conf, conf["tid2pdf"]), dtype="<i4")
    gold = [l.rstrip("\n").split("\t") for l in open(os.path.join(here, "..", "toy_decode_ref.txt"))]
    got = host_decode(oracle, graph, tid2pdf, layers, prior, golden["cmvn_stats"],
                      [golden[name + "_pcm"] for name, _, _ in gold])
    for (name, hyp, llpf), (ids, w) in zip(gold, got):
        assert " ".join(mg.TOY_WORDS[i] for i in ids) == hyp.strip(), name
        assert abs(w - float(llpf)) < 1e-5, name


# ---------------------------------------------------------------- live compiled reference
def test_live_reference_random(oracle, reference, golden, tmp_path):
    if reference is None:
        pytest.skip("oracle/_ref not built (no /root/reference here)")
    pcm = synth_pcm(99, [5], 48000)[0].astype(np.float32)
    fb_r = reference.fbank(pcm)
    fb_o = oracle.fbank(pcm)
    assert np.max(np.abs(fb_o - fb_r) / np.abs(fb_r)) < 1e-5
    assert np.array_equal(oracle.cmvn(fb_r, golden["cmvn_stats"]),
                          reference.cmvn(fb_r, golden["cmvn_stats"]))
    x = np.random.default_rng(0).standard_normal(512).astype(np.float32)
    assert rel_err(oracle.srfft(x), reference.srfft(x)) < 5e-6
    # a mid-size net through Nnet::Read / Propagate, incl. a K > 512 layer (two K-chunks)
    rng = np.random.default_rng(3)
    layers = formats.make_dnn(rng, 600, 96, 2, 50, normalize=True)
    path = str(tmp_path / "n.nnet")
    formats.write_nnet(path, layers)
    xin = rng.standard_normal((37, 600)).astype(np.float32)
    y_r = reference.nnet_propagate(path, xin, 50)
    y_o = oracle.nnet(xin, layers)
    assert np.max(np.abs(y_o - y_r)) < 1e-6
    A = rng.random((121, 17), dtype=np.float32)
    B = rng.random((17, 233), dtype=np.float32)
    assert np.max(np.abs(reference.gemm(A, B) - oracle.simple_matmat(A, B))) < 0.01
