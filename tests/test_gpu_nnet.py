"""GPU parity of the nnet / acoustic-model path (tcgen05 GEMMs + fused epilogues) through the
C ABI, against the compiled-reference golden vectors and the restatement oracle."""

import os
import sys

import numpy as np
import pytest

import pocketkaldi_b200 as pk
from pocketkaldi_b200 import formats
from pocketkaldi_b200.synth import synth_pcm

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_gpu_gemm_matrix import C_MODE, PREC_ID, SCALE, make_net, make_prior, needed_c, splice  # noqa: E402

pytestmark = pytest.mark.gpu

LL_TOL = 2e-2        # north_star: log-likelihoods within 2e-2 absolute
ARGMAX_MIN = 0.999   # north_star: per-frame argmax pdf agreement


@pytest.fixture(scope="module")
def ctx():
    c = pk.Context(0)
    yield c
    c.close()


def toy_layers(toy_conf):
    conf = formats.read_conf(toy_conf)
    layers = formats.read_nnet(formats.conf_path(toy_conf, conf["nnet"]))
    prior = formats.read_vector(formats.conf_path(toy_conf, conf["prior"]))
    return conf, layers, prior


def test_nnet_known_answers(ctx, golden):
    # test/nnet_test.cc:23-73 (Linear 3->4 and Softmax known answers; tolerance of the
    # split-BF16 path is 1e-5 instead of the reference's FP32 1e-6)
    W, b, x = golden["nnet_kat_W"], golden["nnet_kat_b"], golden["nnet_kat_x"]
    y = pk.Nnet(ctx).from_layers([("linear", W, b)]).Propagate(x)
    assert np.max(np.abs(y - golden["nnet_kat_linear_y"])) < 1e-5
    eye = np.eye(4, dtype=np.float32)
    z = np.zeros(4, np.float32)
    ys = pk.Nnet(ctx).from_layers([("linear", eye, z), ("softmax",)]).Propagate(golden["nnet_kat_x4"])
    assert np.max(np.abs(ys - golden["nnet_kat_softmax_y"])) < 1e-5
    # ReLU and Normalize are only reachable fused behind a linear layer
    yr = pk.Nnet(ctx).from_layers([("linear", eye, z), ("relu",), ("linear", eye, z)]).Propagate(golden["nnet_kat_x4"])
    assert np.max(np.abs(yr - golden["nnet_kat_relu_y"])) < 1e-5
    yn = pk.Nnet(ctx).from_layers([("linear", eye, z), ("normalize",), ("linear", eye, z)]).Propagate(golden["nnet_kat_x4"])
    assert abs(float((yn.astype(np.float64) ** 2).sum()) - 4.0) < 1e-4


@pytest.mark.parametrize("m,n,k", [(512, 512, 512), (100, 100, 1), (1, 1, 1), (121, 233, 17),
                                   (300, 3000, 1024), (1000, 1024, 440)])
def test_gemm_differential(ctx, oracle, m, n, k):
    # test/gemm_test.cc:32-62 shapes (+ the config-3 layer shapes): linear layer vs the oracle
    rng = np.random.default_rng(m + n + k)
    A = rng.random((m, k), dtype=np.float32)
    W = rng.random((n, k), dtype=np.float32)
    b = rng.standard_normal(n).astype(np.float32)
    ref = A.astype(np.float64) @ W.astype(np.float64).T + b
    y3 = pk.Nnet(ctx, pk.PREC_BF16X3).from_layers([("linear", W, b)]).Propagate(A)
    assert y3.shape == (m, n)
    assert np.max(np.abs(y3 - ref) / np.maximum(1.0, np.abs(ref))) < 2e-5
    y1 = pk.Nnet(ctx, pk.PREC_BF16).from_layers([("linear", W, b)]).Propagate(A)
    assert np.max(np.abs(y1 - ref) / np.maximum(1.0, np.abs(ref))) < 1e-2
    yh = pk.Nnet(ctx, pk.PREC_FP16X3).from_layers([("linear", W, b)]).Propagate(A)
    assert np.max(np.abs(yh - ref) / np.maximum(1.0, np.abs(ref))) < 2e-6 * max(1.0, k ** 0.5)
    if m * n * k <= 512 ** 3:
        yo = oracle.linear(A, W, b)
        assert np.max(np.abs(y3 - yo) / np.maximum(1.0, np.abs(yo))) < 2e-5


@pytest.mark.parametrize("name", ["hello", "cat", "noise10"])
def test_am_loglik_vs_reference_golden(ctx, golden, toy_conf, name):
    am = pk.AcousticModel(ctx, pk.PREC_BF16X3).Read(toy_conf)
    assert am.num_pdfs() == 12
    ll = am.Compute(golden[name + "_cmvn_ref"])
    ref = golden[name + "_toy_loglik_ref"]
    assert ll.shape == ref.shape
    assert np.max(np.abs(ll - ref)) < LL_TOL
    assert np.mean(ll.argmax(1) == ref.argmax(1)) >= ARGMAX_MIN


def test_decodable_vs_reference_golden(ctx, golden, toy_conf):
    am = pk.AcousticModel(ctx, pk.PREC_BF16X3).Read(toy_conf)
    d = pk.Decodable(am, 0.1, golden["hello_cmvn_ref"])
    ref = golden["hello_toy_decodable_ref"]
    got = np.array([[d.loglikelihood(t, tid) for tid in range(1, 25)] for t in range(ref.shape[0])],
                   np.float32)
    assert np.max(np.abs(got - ref)) < LL_TOL * 0.1
    assert [d.islastframe(t) for t in range(ref.shape[0])] == [bool(v) for v in golden["hello_toy_islast_ref"]]
    assert am.TransitionIdToPdfId(3) == 1 and am.TransitionIdToPdfId(9999) == -1


def test_am_batch_ragged_matches_single(ctx, golden, toy_conf, oracle):
    conf, layers, prior = toy_layers(toy_conf)
    am = pk.AcousticModel(ctx, pk.PREC_BF16X3).Read(toy_conf)
    rng = np.random.default_rng(4)
    feats = [(rng.standard_normal((n, 40)) * 2.5).astype(np.float32) for n in (1, 0, 7, 130, 3, 257)]
    outs = am.compute_batch(feats)
    for f, o in zip(feats, outs):
        assert o.shape == (f.shape[0], 12)
        if f.shape[0]:
            ref = oracle.am_compute(f, layers, prior, 5, 5)
            assert np.max(np.abs(o - ref)) < LL_TOL
            assert np.array_equal(o, am.Compute(f))


@pytest.mark.parametrize("normalize", [False, True])
def test_mid_size_dnn_vs_oracle(ctx, oracle, normalize):
    # 440 -> 3 x 256 -> 1000, random init (SURVEY.md 8d distribution), 600 frames, ragged batch
    rng = np.random.default_rng(11)
    layers = formats.make_dnn(rng, 440, 256, 3, 1000, normalize=normalize)
    prior = np.full(1000, 1e-3, np.float32)
    feats = [(rng.standard_normal((n, 40)) * 2.5).astype(np.float32) for n in (250, 350)]
    ref = [oracle.am_compute(f, layers, prior, 5, 5) for f in feats]
    am3 = pk.AcousticModel(ctx, pk.PREC_BF16X3).from_layers(layers, prior, 5, 5)
    for o, r in zip(am3.compute_batch(feats), ref):
        assert np.max(np.abs(o - r)) < LL_TOL
        assert np.mean(o.argmax(1) == r.argmax(1)) >= ARGMAX_MIN
    # plain BF16 (throughput mode): looser, reported rather than gated at the parity bar
    am1 = pk.AcousticModel(ctx, pk.PREC_BF16).from_layers(layers, prior, 5, 5)
    for o, r in zip(am1.compute_batch(feats), ref):
        assert np.max(np.abs(o - r)) < 0.5
        assert np.mean(o.argmax(1) == r.argmax(1)) >= 0.9


@pytest.mark.parametrize("normalize", [False, True])
@pytest.mark.parametrize("prec", ["PREC_FP16C8", "PREC_FP16X3"])
def test_fp8_corrected_and_split_fp16_modes_vs_oracle(ctx, oracle, prec, normalize):
    # FP16C8 (FP16 product + FP8 first-order corrections, operand mode 3 from the second layer on)
    # and FP16X3 on a 4-layer net with odd widths: hidden 320 (block_n 128 + K tail of the FP8
    # k-blocks), 512 (block_n 256, CTA pairs), 1000 pdfs; ragged batch
    rng = np.random.default_rng(23)
    layers = []
    d = 440
    for o in (320, 512, 256):
        layers += [("linear", (rng.standard_normal((o, d)) * np.sqrt(2.0 / d)).astype(np.float32),
                    (rng.standard_normal(o) * 0.1).astype(np.float32)), ("relu",)]
        if normalize:
            layers.append(("normalize",))
        d = o
    layers += [("linear", (rng.standard_normal((1000, d)) * np.sqrt(2.0 / d)).astype(np.float32),
                (rng.standard_normal(1000) * 0.1).astype(np.float32)), ("softmax",)]
    prior = rng.uniform(0.5, 1.5, 1000).astype(np.float32)
    prior /= prior.sum()
    feats = [(rng.standard_normal((n, 40)) * 2.5).astype(np.float32) for n in (300, 1, 420)]
    ref = [oracle.am_compute(f, layers, prior, 5, 5) for f in feats]
    am = pk.AcousticModel(ctx, getattr(pk, prec)).from_layers(layers, prior, 5, 5)
    worst = 0.0
    for o, r in zip(am.compute_batch(feats), ref):
        worst = max(worst, float(np.max(np.abs(o - r))))
        assert np.mean(o.argmax(1) == r.argmax(1)) >= ARGMAX_MIN
    am.close()
    print(prec, "max |dLL|", worst)
    # both are far inside the 2e-2 bar: ~2^-15 relative for FP16C8, FP32-class for FP16X3
    assert worst < (2e-3 if prec == "PREC_FP16C8" else 2e-4)


def test_fp16c8_linear_layers_alone(ctx):
    # operand mode 3 in isolation: two linear layers (the second one runs FP16 + FP8 corrections)
    # against float64, with weights and activations of very different magnitudes per layer
    rng = np.random.default_rng(3)
    for scale_w, scale_a, k, n in ((0.03, 1.0, 1024, 512), (4.0, 0.02, 200, 130), (1e-3, 30.0, 640, 1024)):
        W1 = np.eye(k, dtype=np.float32)
        b1 = np.zeros(k, np.float32)
        W2 = (rng.standard_normal((n, k)) * scale_w).astype(np.float32)
        b2 = rng.standard_normal(n).astype(np.float32)
        A = np.abs(rng.standard_normal((257, k)) * scale_a).astype(np.float32)
        ref = A.astype(np.float64) @ W2.astype(np.float64).T + b2
        y8 = pk.Nnet(ctx, pk.PREC_FP16C8).from_layers([("linear", W1, b1), ("linear", W2, b2)]).Propagate(A)
        y1 = pk.Nnet(ctx, pk.PREC_FP16).from_layers([("linear", W1, b1), ("linear", W2, b2)]).Propagate(A)
        norm = np.sqrt((A.astype(np.float64) ** 2) @ (W2.astype(np.float64).T ** 2))  # sqrt(sum (a w)^2)
        e8 = float(np.max(np.abs(y8 - ref) / norm))
        e1 = float(np.max(np.abs(y1 - ref) / norm))
        print("k=%d n=%d: fp16c8 %.2e, fp16 %.2e (relative to the product norm)" % (k, n, e8, e1))
        assert e8 < 1.5e-4 and e8 < e1 / 4


def test_model_creation_is_reproducible(ctx):
    # regression: the FP16C8 weight planes of small layers were once packed from a staging buffer
    # whose upload had not landed yet (pageable cudaMemcpy + a non-blocking stream); every instance
    # of the same model must give bit-identical results
    rng = np.random.default_rng(23)
    layers = formats.make_dnn(rng, 440, 320, 1, 1000)
    prior = np.full(1000, 1e-3, np.float32)
    feats = [(rng.standard_normal((n, 40)) * 2.5).astype(np.float32) for n in (300, 1, 420)]
    first = None
    for prec in (pk.PREC_FP16C8, pk.PREC_BF16X3):
        first = None
        for _ in range(6):
            am = pk.AcousticModel(ctx, prec).from_layers(layers, prior, 5, 5)
            outs = am.compute_batch(feats)
            am.close()
            if first is None:
                first = outs
            else:
                assert all(np.array_equal(a, b) for a, b in zip(first, outs))


def test_fused_pcm_to_loglik(ctx, golden, toy_conf):
    am = pk.AcousticModel(ctx, pk.PREC_BF16X3).Read(toy_conf)
    pcms = [golden["hello_pcm"], golden["cat_pcm"], synth_pcm(1234, [0], 160000)[0],
            np.zeros(100, np.int16)]
    lls, feats = am.pcm_to_loglik(pcms, golden["cmvn_stats"], 1.0, want_feats=True)
    for name, ll, ft in zip(["hello", "cat", "noise10"], lls, feats):
        assert np.max(np.abs(ft - golden[name + "_cmvn_ref"]) /
                      np.maximum(1.0, np.abs(golden[name + "_cmvn_ref"]))) < 1e-4
        ref = golden[name + "_toy_loglik_ref"]
        assert np.max(np.abs(ll - ref)) < LL_TOL
        assert np.mean(ll.argmax(1) == ref.argmax(1)) >= ARGMAX_MIN
    assert lls[3].shape == (0, 12)


def test_unsupported_stack_is_an_error(ctx):
    with pytest.raises(pk.PkbError) as e:
        pk.Nnet(ctx).from_layers([("relu",), ("linear", np.eye(4, dtype=np.float32), np.zeros(4, np.float32))])
    assert e.value.code == 5


def test_fp16_mode_meets_loglik_tolerance(ctx, oracle):
    # FP16 operands: BF16 tensor throughput with an 11-bit significand. On the random-init
    # 440 -> 3x256 -> 1000 net the log-likelihood tolerance holds; argmax agreement is reported
    # against the 99.9 % bar separately in DESIGN.md (near-ties flip).
    rng = np.random.default_rng(11)
    layers = formats.make_dnn(rng, 440, 256, 3, 1000)
    prior = np.full(1000, 1e-3, np.float32)
    feats = [(rng.standard_normal((n, 40)) * 2.5).astype(np.float32) for n in (250, 350)]
    ref = [oracle.am_compute(f, layers, prior, 5, 5) for f in feats]
    am = pk.AcousticModel(ctx, pk.PREC_FP16).from_layers(layers, prior, 5, 5)
    for o, r in zip(am.compute_batch(feats), ref):
        assert np.max(np.abs(o - r)) < LL_TOL
        assert np.mean(o.argmax(1) == r.argmax(1)) >= 0.99


@pytest.mark.parametrize("in_ctx,hidden,n_hidden,pdfs,normalize", [
    ((0, 0), 8, 1, 10, False),      # tiny, P % 4 != 0 -> scalar output path, no splice
    ((1, 2), 100, 2, 7, True),      # asymmetric context, odd sizes, normalize
    ((5, 5), 130, 1, 129, False),   # N just above one 128-tile
    ((3, 3), 260, 2, 257, True),    # N just above one 256-tile
    ((5, 5), 64, 0, 300, False),    # single linear + softmax
])
def test_odd_shapes_vs_oracle(ctx, oracle, in_ctx, hidden, n_hidden, pdfs, normalize):
    left, right = in_ctx
    rng = np.random.default_rng(hidden * 1000 + pdfs)
    layers = formats.make_dnn(rng, 40 * (left + right + 1), hidden, n_hidden, pdfs, normalize=normalize)
    prior = rng.uniform(0.5, 1.5, pdfs).astype(np.float32)
    prior /= prior.sum()
    feats = [(rng.standard_normal((n, 40)) * 2.5).astype(np.float32) for n in (1, 129, 2, 300)]
    am = pk.AcousticModel(ctx, pk.PREC_BF16X3).from_layers(layers, prior, left, right)
    outs = am.compute_batch(feats, 0.1)
    for f, o in zip(feats, outs):
        ref = oracle.decodable(f, layers, prior, left, right, 0.1)
        assert o.shape == ref.shape
        assert np.max(np.abs(o - ref)) < LL_TOL * 0.1
        assert np.mean(o.argmax(1) == ref.argmax(1)) >= ARGMAX_MIN


def test_nnet_propagate_without_softmax_and_odd_input_dim(ctx, oracle):
    # Nnet::Propagate on a stack that ends in a linear layer (raw outputs), input dim 37
    rng = np.random.default_rng(5)
    layers = formats.make_dnn(rng, 37, 50, 1, 21)[:-1]
    x = rng.standard_normal((77, 37)).astype(np.float32)
    y = pk.Nnet(ctx).from_layers(layers).Propagate(x)
    ref = oracle.nnet(x, layers)
    assert y.shape == ref.shape == (77, 21)
    assert np.max(np.abs(y - ref)) < 1e-4


@pytest.mark.parametrize("prec", ["bf16x3", "fp16c8"])
def test_spliced_rows_with_unaligned_feat_dim_vs_float64(ctx, prec):
    # feat_dim 13 is not a multiple of 8, so layer 0 is stored with 16 columns per context frame and
    # pkb_nnet_propagate has to pack its 65-column rows in that layout. Nnet has no context, so the
    # model is an AcousticModel passed to pkb_nnet_propagate directly.
    rng = np.random.default_rng(13)
    layers = make_net(rng, (65, 256, 300))
    prior = make_prior(rng, 300)
    feats = (rng.standard_normal((300, 13)) * 2.5).astype(np.float32)
    x = splice(feats, 2, 2)
    am = pk.AcousticModel(ctx, PREC_ID[prec]).from_layers(layers, prior, 2, 2)
    try:
        prob = np.empty((300, 300), np.float32)
        rc = ctx.lib.pkb_nnet_propagate(ctx.h, am.h, x, 300, 65, prob)
        assert rc == 0, ctx.lib.pkb_last_error().decode()
        loglik = am.compute_batch([feats], SCALE)[0]
    finally:
        am.close()
    for out, got in (("prob", prob), ("loglik", loglik)):
        c, _ = needed_c(prec, out, got, x, layers, prior)
        assert c <= C_MODE[prec], "%s %s: error needs c = %.3g > %.3g" % (prec, out, c, C_MODE[prec])


def test_config3_size_properties(ctx, golden):
    # config-3 net on 48 x 10 s through the device-resident pipeline: size-independent
    # properties instead of a CPU oracle -- (1) posteriors renormalise: sum_p prior_p *
    # exp(ll_p / scale) == 1 per frame, (2) utterances are independent: the same utterance ids
    # give the same bits at other batch positions, (3) BF16X3 vs FP16 vs BF16 orderings agree
    rng = np.random.default_rng(0)
    layers = formats.make_dnn(rng, 440, 1024, 6, 3000)
    prior = rng.uniform(0.5, 1.5, 3000).astype(np.float32)
    prior /= prior.sum()
    n_utts, n = 48, 160000
    scale = 0.1
    outs = {}
    for name, prec in (("bf16x3", pk.PREC_BF16X3), ("fp16", pk.PREC_FP16), ("bf16", pk.PREC_BF16)):
        am = pk.AcousticModel(ctx, prec).from_layers(layers, prior, 5, 5)
        b = pk.Batch(ctx, [n] * n_utts, golden["cmvn_stats"], am, prob_scale=scale)
        b.synth_pcm(1234, 0)
        b.run(pk.STAGE_ALL)
        ll = b.get(pk.BUF_LOGLIK).reshape(n_utts, 998, 3000)
        assert np.isfinite(ll).all()
        post = np.exp(ll.astype(np.float64) / scale) * prior.astype(np.float64)
        tol = {"bf16x3": 1e-4, "fp16": 1e-4, "bf16": 1e-4}[name]
        assert np.max(np.abs(post.sum(axis=2) - 1.0)) < tol
        b2 = pk.Batch(ctx, [n] * 3, golden["cmvn_stats"], am, prob_scale=scale)
        b2.synth_pcm(1234, 20)
        b2.run(pk.STAGE_ALL)
        assert np.array_equal(b2.get(pk.BUF_LOGLIK).reshape(3, 998, 3000), ll[20:23])
        chk = b.checksum(pk.BUF_LOGLIK)
        assert abs(chk - float(ll.astype(np.float64).sum())) < 1e-6 * abs(chk)
        outs[name] = ll
        b.close()
        b2.close()
        am.close()
    # single-MMA modes against the parity mode over 47 904 frames x 3000 pdfs. With the speech
    # CMVN statistics applied to synthetic noise the features (and activations) are larger than in
    # the bench distribution and the FP16 tail maximum (observed 4.6e-2 unscaled) exceeds the 2e-2
    # bar it meets there (tools/precision_stats.py: 9e-3); bounded here, reported in DESIGN.md.
    ref = outs["bf16x3"]
    d16 = np.abs(outs["fp16"] - ref) / scale
    assert d16.max() < 1e-1 and d16.mean() < 5e-3
    assert np.mean(outs["fp16"].argmax(2) == ref.argmax(2)) > 0.995
    assert np.abs(outs["bf16"] - ref).max() / scale < 1.0
    assert np.mean(outs["bf16"].argmax(2) == ref.argmax(2)) > 0.97


def test_loader_errors_follow_the_reference_convention(ctx, tmp_path, toy_conf):
    # AcousticModel::Read error classes (src/am.cc:23-63, src/status.h:37-100): missing file ->
    # IOError, malformed section -> Corruption, missing key -> Corruption "Unable to find key"
    with pytest.raises(pk.PkbError) as e:
        pk.AcousticModel(ctx).Read(str(tmp_path / "nope.conf"))
    assert e.value.code == 2 and "IOError" in str(e.value)
    import shutil
    # contents only: copied modes would leave the copies read-only where the test tree is
    src = os.path.dirname(toy_conf)
    d = tmp_path / "m"
    d.mkdir()
    for f in os.listdir(src):
        shutil.copyfile(os.path.join(src, f), d / f)
    conf = str(d / "toy.conf")
    raw = bytearray(open(d / "toy.nnet", "rb").read())
    raw[0:4] = b"XXXX"
    open(d / "toy.nnet", "wb").write(bytes(raw))
    with pytest.raises(pk.PkbError) as e:
        pk.AcousticModel(ctx).Read(conf)
    assert e.value.code == 3 and "Corruption" in str(e.value)
    shutil.copyfile(os.path.join(src, "toy.nnet"), d / "toy.nnet")
    lines = [l for l in open(conf) if not l.startswith("prior")]
    open(conf, "w").writelines(lines)
    with pytest.raises(pk.PkbError) as e:
        pk.AcousticModel(ctx).Read(conf)
    assert e.value.code == 3 and "Unable to find key 'prior'" in str(e.value)
    # unknown layer types are rejected like the reference reader does (src/nnet.cc:122-126);
    # MUL (5) and the optional sigmoid (6, tests/test_gpu_options.py) are the extensions, see
    # test_mul_layers_are_folded_into_linear
    import struct
    for bad_type in (4, 7, -1):
        with open(d / "bad.nnet", "wb") as fd:
            fd.write(b"NNT0" + struct.pack("<ii", 4, 1) + b"LAY0" + struct.pack("<ii", 4, bad_type))
        open(conf, "w").writelines([l.replace("toy.nnet", "bad.nnet") if l.startswith("nnet") else l
                                    for l in open(toy_conf)])
        with pytest.raises(pk.PkbError) as e:
            pk.AcousticModel(ctx).Read(conf)
        assert e.value.code == 3 and "unexpected layer type: %d" % bad_type in str(e.value)


def test_mul_layers_are_folded_into_linear(ctx, oracle, reference, tmp_path, golden):
    # SURVEY 8(f)-3: tool/convert_am.py writes a MUL layer for Kaldi's FixedScaleComponent; the
    # reference reader rejects such a model, libpkb200 folds y = x * v into the neighbouring
    # LinearLayer when it loads the file. Checked against the oracle on the hand-folded model
    # (tight) and against a float64 evaluation of the unfolded layer list (the semantics).
    rng = np.random.default_rng(11)
    base = formats.make_dnn(rng, 440, 96, 2, 24, normalize=True)
    v_in = rng.uniform(0.5, 1.5, 440).astype(np.float32)
    v_h = rng.uniform(-1.5, 1.5, 96).astype(np.float32)      # negative scales are fine before ReLU
    v_out = rng.uniform(0.2, 3.0, 24).astype(np.float32)
    layers = [("mul", v_in)]
    n_lin = 0
    for l in base:
        layers.append(l)
        if l[0] == "linear":
            n_lin += 1
            if n_lin == 1:
                layers.append(("mul", v_h))
            if n_lin == 3:
                layers += [("mul", v_out), ("mul", np.full(24, 0.5, np.float32))]
    prior = rng.dirichlet(np.ones(24)).astype(np.float32)
    conf = formats.write_model_dir(str(tmp_path), "mul", layers, prior, 5, 5, list(range(24)),
                                   cmvn_stats=golden["cmvn_stats"])
    assert [l[0] for l in formats.read_nnet(str(tmp_path / "mul.nnet"))].count("mul") == 4
    if reference is not None:
        with pytest.raises(Exception):
            reference.am_load(conf)
    am = pk.AcousticModel(ctx, pk.PREC_BF16X3).Read(conf)
    feats = golden["hello_cmvn_ref"]
    got = am.Compute(feats)
    folded = formats.fold_mul_layers(layers)
    assert all(l[0] != "mul" for l in folded) and len(folded) == len(base)
    want = oracle.am_compute(feats, folded, prior, 5, 5)
    assert np.max(np.abs(got - want)) < 2e-3
    assert np.mean(got.argmax(1) == want.argmax(1)) >= 0.999

    def forward64(x):
        T = x.shape[0]
        idx = np.clip(np.arange(T)[:, None] + np.arange(-5, 6)[None, :], 0, T - 1)
        h = x.astype(np.float64)[idx].reshape(T, -1)
        for l in layers:
            if l[0] == "mul":
                h = h * l[1].astype(np.float64)
            elif l[0] == "linear":
                h = h @ l[1].astype(np.float64).T + l[2]
            elif l[0] == "relu":
                h = np.maximum(h, 0)
            elif l[0] == "normalize":
                h = h * np.sqrt(h.shape[1] / np.sum(h * h, axis=1, keepdims=True))
            else:
                e = np.exp(h - h.max(1, keepdims=True))
                h = e / e.sum(1, keepdims=True)
        return np.log(np.maximum(h, 1e-20)) - np.log(prior.astype(np.float64))
    assert np.max(np.abs(got - forward64(feats))) < 2e-3

    # a MUL that is not next to a linear layer cannot be folded
    bad = [base[0], base[1], ("mul", np.ones(96, np.float32))] + base[2:]
    conf2 = formats.write_model_dir(str(tmp_path), "mul2", bad, prior, 5, 5, list(range(24)),
                                    cmvn_stats=golden["cmvn_stats"])
    with pytest.raises(pk.PkbError) as e:
        pk.AcousticModel(ctx).Read(conf2)
    assert e.value.code == 5
    with pytest.raises(ValueError):
        formats.fold_mul_layers(bad)


def test_lazy_decodable_matches_eager_bitwise(ctx, golden, toy_conf):
    # SURVEY 8(f)-1 through the C ABI: pkb_am_compute_chunked + pkb_event_*
    am = pk.AcousticModel(ctx, pk.PREC_BF16X3).Read(toy_conf)
    feats = golden["cat_cmvn_ref"]
    eager = pk.Decodable(am, 0.1, feats)
    for chunk in (1, 7, 64, 10 ** 6):
        lazy = pk.Decodable(am, 0.1, feats, chunk_frames=chunk)
        T = feats.shape[0]
        # frame-synchronous access like Decoder::ProcessEmitting
        for t in (0, 1, T // 2, T - 1):
            for tid in (1, 5):
                assert lazy.loglikelihood(t, tid) == eager.loglikelihood(t, tid)
        assert lazy.islastframe(T - 1) and not lazy.islastframe(0)
        assert lazy.frames_ready() == T
        assert np.array_equal(np.asarray(lazy.log_prob), eager.log_prob)
        lazy.close()
    # an early frame does not need the whole matrix
    lazy = pk.Decodable(am, 0.1, feats, chunk_frames=16)
    lazy.loglikelihood(0, 1)
    assert 16 <= lazy._ready <= feats.shape[0]
    lazy.close()
    # no frames
    empty = pk.Decodable(am, 0.1, np.zeros((0, 40), np.float32), chunk_frames=8)
    assert empty.log_prob.shape == (0, am.num_pdfs())
    empty.close()
