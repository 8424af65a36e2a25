"""Every tcgen05 GEMM variant and every output mode against a float64 forward pass.

launch_gemm (pocketkaldi_b200/csrc/gemm_sm100.cu) instantiates gemm_kernel<BN, PLANES, FINAL, CG,
OUT8> for each PKB_GEMM_CASE, and nnet_forward (nnet.cu) picks one per stage from the layer
widths, the row count and the precision. The case table below reaches all of them;
test_case_table_reaches_every_gemm_variant (no GPU) checks that with a Python mirror of those
dispatch rules, so a variant added later fails it until the table covers it.

Error bounds. forward64 returns the logits z and their magnitude m = |W_L| a_{L-1}, the part that
went through 16-bit operands (a_l = |W_l| a_{l-1} + |b_l|, with a sigmoid adding its output and
scaling a by 1/4, and a normalize scaling it by the reference row scale; the last bias is added in
FP32). A logit is within delta = c * u * m + 2^-21 |z|, with u the operand unit of the precision
plus FP32 accumulation over the widest fan-in K (K * 2^-24). Each output mode carries
delta over: loglik <= 2 s delta_row, prob <= p (e^{2 delta_row} - 1), compact adds half an fp16
ulp of t - off. Each check computes the smallest c that covers every element and asserts it is
below C_MODE. Each multi-term mode must also be at least 4x more accurate than its single-term
counterpart on the same case, so a dropped lo plane or FP8 correction phase fails.
"""

import os
import re

import numpy as np
import pytest

import pocketkaldi_b200 as pk
from pocketkaldi_b200.synth import synth_global_cmvn, synth_pcm

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GEMM_SRC = os.path.join(ROOT, "pocketkaldi_b200", "csrc", "gemm_sm100.cu")
B200_SMS = 148
SCALE = 0.1
LOG_FLOOR = float(np.log(np.float64(np.float32(1e-20))))

PRECS = ("bf16", "fp16", "bf16x3", "fp16x3", "fp16c8")
PREC_ID = {"bf16": pk.PREC_BF16, "fp16": pk.PREC_FP16, "bf16x3": pk.PREC_BF16X3,
           "fp16x3": pk.PREC_FP16X3, "fp16c8": pk.PREC_FP16C8, "fp16r": pk.PREC_FP16R}
# operand unit of each precision: BF16 / FP16 significands, their hi+lo splits, and FP16C8
# (FP16 product + the two first-order corrections through E4M3)
U_MODE = {"bf16": 2.0 ** -8, "fp16": 2.0 ** -11, "bf16x3": 2.0 ** -16, "fp16x3": 2.0 ** -22,
          "fp16c8": 2.0 ** -15}
# Largest c (see the module docstring) a check may need: about 3x the largest c measured over all
# cases of this file (printed as CALIBRATION lines with -s) on an NVIDIA B200 at a 1000 W power
# limit. Measured maxima, all on the K = 1 net in raw mode: bf16 0.272, fp16 0.278, bf16x3 0.0759,
# fp16x3 0.0165, fp16c8 0.0861; the deep nets of the matrix need 1e-3 or less. With the sigmoid
# padding columns left in the normalize sum, the width-200 sigmoid net needed bf16x3 3.61,
# fp16x3 5.67 and fp16c8 2.64.
C_MODE = {"bf16": 0.8, "fp16": 0.8, "bf16x3": 0.25, "fp16x3": 0.05, "fp16c8": 0.25}
MULTI_TERM = (("bf16x3", "bf16"), ("fp16x3", "fp16"), ("fp16c8", "fp16"))
OUTS = ("raw", "prob", "loglik", "compact")

# ------------------------------------------------------------------------------ the case table
# net A: hidden 512 (block_n 256) then 320 (128), 1000 pdfs (256). net B: hidden 320 (128) then
# 512 (256), 300 pdfs (128, 3 tiles). M = 97 is one row tile (no CTA pairs); M = 300 is an odd
# tile count, so the CTA of the last pair works past the end.
NET_A = (440, 512, 320, 1000)
NET_B = (440, 320, 512, 300)
MATRIX = [(net, m, out) for net in (NET_A, NET_B) for m in (97, 300) for out in OUTS]
# 79 column tiles of 256: more than the 74 SM pairs, so the softmax stage drops to cta_group 1
WIDE = [("bf16x3", (440, 256, 20000), 300, "loglik"), ("fp16c8", (440, 256, 20000), 300, "loglik")]


def case_table():
    """(precision, dims, M, output mode) of every GEMM case this file runs."""
    return [(p, net, m, out) for net, m, out in MATRIX for p in PRECS] + WIDE


# ---------------------------------------------------------------- dispatch mirror (no GPU)
def block_n(n):
    """alloc_stage: 256-wide tiles unless they cost more than 6 % extra padding (nnet.cu:124)."""
    n128, n256 = -(-n // 128) * 128, -(-n // 256) * 256
    return 256 if n256 * 100 <= n128 * 106 else 128


def launched(prec, dims, m, out, selected=None, sms=B200_SMS):
    """The (BN, PLANES, FINAL, CG, OUT8) instantiations nnet_forward launches for a net of widths
    `dims` on m rows. FP16R log-likelihoods run a one-MMA pass over every row and the FP16C8
    operands over `selected` rows (nnet_forward_refined)."""
    c8 = prec in ("fp16c8", "fp16r")
    planes = 2 if prec in ("bf16x3", "fp16x3") or c8 else 1
    if prec == "fp16r" and out in ("loglik", "compact"):
        passes = [(True, m), (False, m if selected is None else selected)]
    else:
        passes = [(False, m)]
    got = set()
    for fast, rows in passes:
        if rows == 0:
            continue
        m_tiles = -(-rows // 128)
        n_stages = len(dims) - 1
        for i in range(n_stages):
            n, final = dims[i + 1], i == n_stages - 1
            bn = block_n(n)
            mode = 1 if fast else (3 if c8 and i > 0 else planes)             # nnet.cu:361
            out8 = not fast and not final and c8                                # nnet.cu:362
            want_pair = not final or mode >= 2                                # nnet.cu:424
            cg = 2 if want_pair and bn == 256 and m_tiles >= 2 else 1
            tiles = -(-n // bn)
            if final and out != "raw" and cg == 2 and (sms // 2) // tiles < 1:  # nnet.cu:427
                cg = 1
            got.add((bn, mode, final, cg, out8))
    return got


def compiled_variants():
    """The PKB_GEMM_CASE(...) list of launch_gemm."""
    pat = re.compile(r"^\s*PKB_GEMM_CASE\((\d+),\s*(\d+),\s*(true|false),\s*(\d+),\s*(true|false)\)")
    cases = set()
    for line in open(GEMM_SRC):
        if line.lstrip().startswith("#define"):
            continue
        mt = pat.match(line)
        if mt:
            bn, pl, fin, cg, o8 = mt.groups()
            cases.add((int(bn), int(pl), fin == "true", int(cg), o8 == "true"))
    return cases


def test_case_table_reaches_every_gemm_variant():
    compiled = compiled_variants()
    assert len(compiled) == 20
    reached = set()
    for case in case_table():
        got = launched(*case)
        assert got <= compiled, "mirror launches a variant launch_gemm does not have: %s" % (got - compiled)
        reached |= got
    missing = sorted(compiled - reached)
    assert not missing, "no case reaches PKB_GEMM_CASE%s" % ", ".join(
        "(%d, %d, %s, %d, %s)" % (bn, pl, str(f).lower(), cg, str(o).lower()) for bn, pl, f, cg, o in missing)


def test_dispatch_mirror_known_answers():
    # the rules the mirror restates, on shapes whose dispatch the nnet.cu comments spell out
    assert [block_n(n) for n in (1, 129, 200, 257, 300, 320, 512, 1000, 3000, 20000)] == \
        [128, 256, 256, 128, 128, 128, 256, 256, 256, 256]
    assert launched("bf16", (440, 1024, 3000), 1000, "loglik") == {(256, 1, False, 2, False), (256, 1, True, 1, False)}
    assert launched("bf16x3", (440, 1024, 3000), 1000, "loglik") == {(256, 2, False, 2, False), (256, 2, True, 2, False)}
    assert launched("bf16x3", (440, 256, 20000), 1000, "loglik") == {(256, 2, False, 2, False), (256, 2, True, 1, False)}
    assert launched("bf16x3", (440, 256, 20000), 1000, "raw") == {(256, 2, False, 2, False), (256, 2, True, 2, False)}
    assert launched("fp16r", (440, 1024, 1024, 3000), 1000, "loglik", selected=100) == {
        (256, 1, False, 2, False), (256, 1, True, 1, False),        # pass 1 over every row
        (256, 2, False, 1, True), (256, 3, False, 1, True), (256, 3, True, 1, False)}  # 100 rows


# ------------------------------------------------------------------ float64 reference
def splice(feats, left, right):
    T = feats.shape[0]
    idx = np.clip(np.arange(T)[:, None] + np.arange(-left, right + 1)[None, :], 0, T - 1)
    return feats[idx].reshape(T, -1)


def forward64(x, layers):
    """(z, m_prod) of the last linear layer of `layers` on input rows x (module docstring)."""
    h = np.asarray(x, np.float64)
    a = np.abs(h)
    mp = None
    for l in layers:
        kind = l[0]
        if kind == "linear":
            W, b = l[1].astype(np.float64), l[2].astype(np.float64)
            h = h @ W.T + b
            mp = a @ np.abs(W).T
            a = mp + np.abs(b)
        elif kind == "relu":
            h = np.maximum(h, 0.0)
        elif kind == "sigmoid":
            h = 1.0 / (1.0 + np.exp(-h))
            a = h + a / 4
        elif kind == "normalize":
            rs = np.sqrt(h.shape[1] / np.sum(h * h, axis=1, keepdims=True))
            h, a = h * rs, a * rs
        elif kind != "softmax":
            raise ValueError(kind)
    return h, mp


def log_softmax64(z):
    zm = z.max(1, keepdims=True)
    return z - zm - np.log(np.exp(z - zm).sum(1, keepdims=True))


def log_prior64(prior):
    # the library stores log(double(prior)) as float (src/am.cc:42-43)
    return np.log(prior.astype(np.float64)).astype(np.float32).astype(np.float64)


def unit(prec, layers):
    k = max(l[1].shape[1] for l in layers if l[0] == "linear")
    return U_MODE["fp16c8" if prec == "fp16r" else prec] + k * 2.0 ** -24


def needed_c(prec, out, got, x, layers, prior=None):
    """(smallest c whose bound covers every element, error measure for the multi-term check)."""
    z, mp = forward64(x, layers)
    got = got.astype(np.float64)
    du = unit(prec, layers) * mp                      # per-unit-c logit error
    fp = 2.0 ** -21 * np.abs(z)                       # FP32 epilogue (bias, row scale, softmax)
    d1 = np.maximum(du.max(1, keepdims=True), 1e-300)
    f1 = fp.max(1, keepdims=True)
    if out == "raw":
        err = np.abs(got - z)
        c = np.maximum(err - fp, 0.0) / np.maximum(du, 1e-300)
        return float(c.max()), float(err.max())
    lsm = log_softmax64(z)
    if out == "prob":
        p = np.exp(lsm)
        err = np.abs(got - p)
        slack = p * 2.0 ** -20 + 1e-37
        c = (np.log1p(np.maximum(err - slack, 0.0) / np.maximum(p, 1e-300)) / 2 - f1) / d1
        return float(max(c.max(), 0.0)), float(err.max())
    lp = log_prior64(prior)
    t = np.maximum(lsm, LOG_FLOOR) - lp               # unscaled log-likelihood
    ref = SCALE * t
    err = np.abs(got - ref)
    slack = SCALE * 2.0 ** -21 * (np.abs(lsm) + np.abs(lp) + 1.0)
    if out == "loglik":
        c = ((err - slack) / (2 * SCALE) - f1) / d1
        return float(max(c.max(), 0.0)), float(err.max())
    # compact: fp16(t - off) with off the frame maximum, plus the rounding of that half
    q = SCALE * (np.abs(t - t.max(1, keepdims=True)) * 2.0 ** -11 + 2.0 ** -25)
    c = ((err - slack - q) / (2 * SCALE * (1 + 2.0 ** -11)) - f1) / d1
    top = np.argmax(ref, axis=1)
    return float(max(c.max(), 0.0)), float(err[np.arange(len(top)), top].max())


# ------------------------------------------------------------------ running the library
def make_net(rng, dims, act="relu", normalize=False):
    layers = []
    for i, (d, o) in enumerate(zip(dims[:-1], dims[1:])):
        layers.append(("linear", (rng.standard_normal((o, d)) * np.sqrt(2.0 / d)).astype(np.float32),
                       (rng.standard_normal(o) * 0.1).astype(np.float32)))
        if i < len(dims) - 2:
            layers.append((act,))
            if normalize:
                layers.append(("normalize",))
    layers.append(("softmax",))
    return layers


def make_prior(rng, n):
    p = rng.uniform(0.5, 1.5, n).astype(np.float32)
    return p / p.sum()


def run_output(ctx, prec, layers, prior, out, feats, left=5, right=5):
    """The library's output for `out` and the spliced input rows the reference starts from.
    raw / prob: Nnet.Propagate; loglik: AcousticModel.compute_batch; compact: a Batch of one
    utterance with as many frames as `feats` has rows, on its own CMVN features."""
    if out in ("raw", "prob"):
        net = layers if out == "prob" else [l for l in layers if l[0] != "softmax"]
        x = splice(feats, left, right)
        nn = pk.Nnet(ctx, PREC_ID[prec]).from_layers(net)
        try:
            return nn.Propagate(x), x
        finally:
            nn.am.close()
    am = pk.AcousticModel(ctx, PREC_ID[prec]).from_layers(layers, prior, left, right)
    try:
        if out == "loglik":
            return am.compute_batch([feats], SCALE)[0], splice(feats, left, right)
        b = pk.Batch(ctx, [400 + 160 * (feats.shape[0] - 1)], synth_global_cmvn(), am, prob_scale=SCALE)
        try:
            b.synth_pcm(77, 0)
            b.run(pk.STAGE_ALL)
            f = b.get(pk.BUF_FEATS)
            b.set_compact(True)
            b.run(pk.STAGE_NNET)
            got = b.expand_compact(b.get(pk.BUF_LOGLIK16), b.get(pk.BUF_LOGLIK_OFF), SCALE)
        finally:
            b.close()
        return got, splice(f, left, right)
    finally:
        am.close()


def check_all_precisions(ctx, label, layers, prior, out, feats, left=5, right=5, precs=PRECS,
                         discriminate=True):
    """Runs `out` in every precision, asserts each bound and the multi-term accuracy margins."""
    errs = {}
    for prec in precs:
        got, x = run_output(ctx, prec, layers, prior, out, feats, left, right)
        assert got.shape == (feats.shape[0], layers[-2][1].shape[0]) and np.isfinite(got).all()
        c, errs[prec] = needed_c(prec, out, got, x, layers, prior)
        print("CALIBRATION %s %s %s c=%.3g err=%.3g" % (label, out, prec, c, errs[prec]))
        assert c <= C_MODE[prec], "%s %s %s: error needs c = %.3g > %.3g" % (label, out, prec, c, C_MODE[prec])
    if discriminate:
        for multi, single in MULTI_TERM:
            if multi in errs and single in errs:
                assert errs[multi] * 4 < errs[single], "%s %s: %s error %.3g is not 4x below %s %.3g" % (
                    label, out, multi, errs[multi], single, errs[single])
    return errs


@pytest.fixture(scope="module")
def ctx():
    c = pk.Context(0)
    yield c
    c.close()


def net_label(dims):
    return "x".join(str(d) for d in dims)


@pytest.mark.gpu
@pytest.mark.parametrize("dims,m,out", MATRIX, ids=["%s-m%d-%s" % (net_label(d), m, o) for d, m, o in MATRIX])
def test_matrix_vs_float64(ctx, dims, m, out):
    rng = np.random.default_rng(sum(dims) + m)
    layers = make_net(rng, dims)
    prior = make_prior(rng, dims[-1])
    feats = (rng.standard_normal((m, 40)) * 2.5).astype(np.float32)
    check_all_precisions(ctx, net_label(dims), layers, prior, out, feats)


@pytest.mark.gpu
@pytest.mark.parametrize("prec,dims,m,out", WIDE, ids=["%s-%s" % (p, net_label(d)) for p, d, _, _ in WIDE])
def test_more_softmax_tiles_than_sm_pairs(ctx, prec, dims, m, out):
    rng = np.random.default_rng(5)
    layers = make_net(rng, dims)
    prior = make_prior(rng, dims[-1])
    feats = (rng.standard_normal((m, 40)) * 2.5).astype(np.float32)
    check_all_precisions(ctx, net_label(dims), layers, prior, out, feats, precs=(prec,))


@pytest.mark.gpu
def test_softmax_tiles_beyond_the_sms_are_rejected(ctx):
    # 157 column tiles of 256 > 148 SMs: launch_gemm refuses before any launch
    rng = np.random.default_rng(8)
    layers = make_net(rng, (440, 256, 40000))
    am = pk.AcousticModel(ctx, pk.PREC_BF16).from_layers(layers, make_prior(rng, 40000), 5, 5)
    try:
        with pytest.raises(pk.PkbError) as e:
            am.compute_batch([(rng.standard_normal((50, 40))).astype(np.float32)], SCALE)
        assert "column tiles exceed" in str(e.value)
    finally:
        am.close()


# ------------------------------------------------------------------ edge rows and columns
def _final(layers, W=None, b=None):
    _, W0, b0 = layers[-2]
    layers[-2] = ("linear", W0 if W is None else W.astype(np.float32), b0 if b is None else b.astype(np.float32))
    return layers


def _edge_n(n):
    return lambda rng: make_net(rng, (440, 256, n))


def _edge_bias_minus50(rng):
    layers = make_net(rng, (440, 256, 300))          # 3 tiles of 128, 84 padding columns
    return _final(layers, b=np.full(300, -50.0))


def _edge_best_in_last_tile(rng):
    layers = make_net(rng, (440, 256, 1001))         # 4 tiles of 256, the last one 233 wide
    b = layers[-2][2].copy()
    b[-1] += 60.0
    return _final(layers, b=b)


def _edge_all_equal(rng):
    layers = make_net(rng, (440, 256, 1001))
    return _final(layers, W=np.zeros_like(layers[-2][1]), b=np.zeros(1001))


def _edge_logits_1e3(rng):
    layers = make_net(rng, (440, 256, 1001))
    return _final(layers, b=1000.0 + rng.standard_normal(1001) * 3.0)


def _edge_floor_binds(rng):
    layers = make_net(rng, (440, 256, 1001))
    return _final(layers, W=layers[-2][1] * 40.0)


EDGES = {"n%d" % n: _edge_n(n) for n in (1, 7, 129, 257, 1001, 1004)}
EDGES.update(bias_minus50=_edge_bias_minus50, best_in_last_tile=_edge_best_in_last_tile,
             all_equal=_edge_all_equal, logits_1e3=_edge_logits_1e3, floor_binds=_edge_floor_binds)
K_TAILS = (1, 63, 64, 65, 127, 129)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(EDGES))
def test_edge_case_vs_float64(ctx, name):
    rng = np.random.default_rng(len(name))
    layers = EDGES[name](rng)
    n = layers[-2][1].shape[0]
    prior = make_prior(rng, n)
    feats = (rng.standard_normal((300, 40)) * 2.5).astype(np.float32)
    x = splice(feats, 5, 5)
    z = forward64(x, layers)[0]
    lsm = log_softmax64(z)
    if name == "best_in_last_tile":
        assert (z.argmax(1) >= 768).all()
    if name == "floor_binds":
        assert (lsm <= LOG_FLOOR).mean() > 0.2
    if name == "logits_1e3":
        assert z.min() > 900
    # a single column, equal logits, a constant bias or one dominant column leave little product
    # error in the softmax outputs, and around 1e3 the FP32 rounding of the logits is as large as
    # the FP16 product error: nothing to tell the precisions apart by
    disc = name not in ("n1", "all_equal", "bias_minus50", "best_in_last_tile", "logits_1e3")
    for out in OUTS:
        check_all_precisions(ctx, name, layers, prior, out, feats, discriminate=disc)
    if name == "all_equal":
        # FP16R: every frame has all pdfs tied, so the second pass recomputes all of them
        am = pk.AcousticModel(ctx, pk.PREC_FP16R).from_layers(layers, prior, 5, 5)
        b = pk.Batch(ctx, [400 + 160 * 299], synth_global_cmvn(), am, prob_scale=SCALE)
        try:
            b.synth_pcm(77, 0)
            b.run(pk.STAGE_ALL)
            assert b.refine_stats() == (300, 300)
            got = b.get(pk.BUF_LOGLIK)
            want = SCALE * (np.log(1.0 / n) - log_prior64(prior))
            assert np.max(np.abs(got - want[None, :])) < 1e-5
        finally:
            b.close()
            am.close()


@pytest.mark.gpu
@pytest.mark.parametrize("k", K_TAILS)
def test_k_tail_vs_float64(ctx, k):
    # input width k: 64-wide K blocks of the 16-bit planes, 128-wide ones of the FP8 planes
    rng = np.random.default_rng(k)
    layers = make_net(rng, (k, 256, 300))
    prior = make_prior(rng, 300)
    feats = (rng.standard_normal((300, k)) * 2.5).astype(np.float32)
    for out in ("raw", "prob", "loglik"):
        check_all_precisions(ctx, "k%d" % k, layers, prior, out, feats, left=0, right=0)


@pytest.mark.gpu
@pytest.mark.parametrize("width", [200, 256])
def test_sigmoid_normalize_vs_float64(ctx, width):
    # width 200 pads to one 256-wide tile: its 56 padding columns must not enter the row's
    # sum of squares (a sigmoid maps their z = 0 to 0.5)
    rng = np.random.default_rng(width)
    layers = make_net(rng, (440, width, width, 300), act="sigmoid", normalize=True)
    prior = make_prior(rng, 300)
    feats = (rng.standard_normal((300, 40)) * 2.5).astype(np.float32)
    for out in ("prob", "loglik"):
        check_all_precisions(ctx, "sigmoid%d" % width, layers, prior, out, feats)


# ------------------------------------------------------------------ the benchmark's own shapes
@pytest.mark.gpu
@pytest.mark.parametrize("config,n_utts", [("3", 4096), ("4", 1024)])
def test_headline_path_at_bench_scale(config, n_utts, oracle):
    """The path bench.py times, at its size (config 3: 4.1 M rows x 3000 pdfs, more than 2^31
    output elements; config 4: 8.2e9 elements, more than 2^32), sampled against float64."""
    import bench
    cfg = bench.CONFIGS[config]
    P, T = cfg["pdfs"], bench.FRAMES_10S
    layers, prior = bench.make_layers(cfg), bench.uniform_prior(cfg)
    g = synth_global_cmvn()
    # utterances holding output element 2^31 (and 2^32) in the padded row layout of the device
    # matrix (pad_off = frame_off + 10 u, one pitch of T + 10 rows) and in the frame layout
    marks = [e for e in (2 ** 31, 2 ** 32) if e < n_utts * T * P]
    focus = {0: None, n_utts - 1: None}
    for e in marks:
        r = e // P
        focus.setdefault(min(r // (T + 10), n_utts - 1), min(r % (T + 10), T - 1))
        focus.setdefault(r // T, r % T)
    rnd = np.random.default_rng(int(config))
    u_pair = int(rnd.integers(1, n_utts - 2))
    for u in (u_pair, u_pair + 1, int(rnd.integers(1, n_utts - 1))):
        focus.setdefault(u, int(rnd.integers(0, T)))
    utts = sorted(focus)
    ctx = pk.Context(0)
    am = pk.AcousticModel(ctx, bench.precision_id(bench.DEFAULT_PRECISION)).from_layers(layers, prior, 5, 5)
    b = None
    try:
        if bench.DEFAULT_PRECISION == "fp16r":
            am.set_refine_margin(bench.REFINE_MARGIN)
        b = pk.Batch(ctx, [bench.SAMPLES_10S] * n_utts, g, am, prob_scale=SCALE)
        b.synth_pcm(1234, 0)
        frames = b.total_frames
        assert frames == n_utts * T
        runs = []
        for _ in range(2):
            b.run(pk.STAGE_ALL | pk.STAGE_NO_FEATS)
            if bench.DEFAULT_PRECISION == "fp16r":
                _, refined = b.refine_stats()
                assert 0 < refined < frames
            rows = {u: np.empty((T, P), np.float32) for u in utts}
            for u in utts:
                b.get_rows_async(pk.BUF_LOGLIK, u * T, T, rows[u])
            pair = np.empty((2 * T, P), np.float32)  # two whole utterances: one strided copy
            b.get_rows_async(pk.BUF_LOGLIK, u_pair * T, 2 * T, pair)
            ctx.sync()
            assert np.array_equal(pair, np.concatenate([rows[u_pair], rows[u_pair + 1]]))
            runs.append(rows)
        for u in utts:
            assert np.array_equal(runs[0][u], runs[1][u]), "utterance %d differs between runs" % u
    finally:
        if b is not None:
            b.close()
        am.close()
        ctx.close()
    flips = n = 0
    worst = 0.0
    for u in utts:
        feats = oracle.cmvn(oracle.fbank(synth_pcm(1234, [u], bench.SAMPLES_10S)[0].astype(np.float32)), g)
        t0, t1 = (0, T) if focus[u] is None else (max(0, focus[u] - 64), min(T, focus[u] + 64))
        z = forward64(splice(feats.astype(np.float64), 5, 5)[t0:t1], layers)[0]
        ref = np.maximum(log_softmax64(z), LOG_FLOOR) - log_prior64(prior)
        got = runs[0][u][t0:t1] / SCALE
        worst = max(worst, float(np.abs(got - ref).max()))
        flips += int(np.sum(got.argmax(1) != ref.argmax(1)))
        n += t1 - t0
    print("config %s: %d utterances sampled, %d frames, max |dLL| %.3g, %d argmax flips" % (
        config, len(utts), n, worst, flips))
    assert worst <= bench.LL_TOL
    assert 1.0 - flips / n >= bench.ARGMAX_MIN
