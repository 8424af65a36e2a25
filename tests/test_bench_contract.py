"""bench.py contract: the reference arm runs without a GPU, prints exactly one JSON line with the
required keys, and times the unmodified reference (oracle/_ref); on the GPU, --dump-outputs
writes what the timed path computed, bounded in size and the same from run to run."""

import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libpkref.so")):
        pytest.skip("oracle/_ref not built")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                          "--config", "2", "--steps", "1", "--warmup", "0"],
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=300, check=True)
    lines = [l for l in out.stdout.decode().splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step",
                "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
                "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["value"] > 0
    assert d["vs_baseline"] is None and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["e2e"]["value"] == d["value"]


def test_reference_arm_nonzero_rank_is_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                          "--config", "2", "--steps", "1", "--warmup", "0", "--gpus", "2"],
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=120, env=env, check=True)
    assert out.stdout.decode().strip() == ""


def run_bench_dump(out_dir, *extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--warmup", "1", "--no-cpu",
                          "--no-e2e", "--no-sub", "--dump-outputs", str(out_dir)] + list(extra),
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600, check=True)
    return json.loads(out.stdout.decode().strip().splitlines()[-1])


@pytest.mark.gpu
def test_dump_outputs_of_the_frontend_config_hold_the_features(tmp_path, oracle):
    import numpy as np
    from pocketkaldi_b200.synth import synth_global_cmvn, synth_pcm
    line = run_bench_dump(tmp_path, "--config", "2", "--utts", "3", "--steps", "2")
    assert line["steps"] == 2
    feats, rows = np.load(tmp_path / "feats.npy"), np.load(tmp_path / "feats_rows.npy")
    assert feats.dtype == np.float32 and feats.shape == (3 * 998, 40)
    assert np.array_equal(rows, np.arange(3 * 998))
    # the batch's first utterance is utterance 0 of the synthetic corpus
    want = oracle.cmvn(oracle.fbank(synth_pcm(1234, [0], 160000)[0].astype(np.float32)), synth_global_cmvn())
    assert np.max(np.abs(feats[:998] - want) / np.maximum(1.0, np.abs(want))) < 1e-4


@pytest.mark.gpu
def test_dump_outputs_sample_is_bounded_and_repeatable(tmp_path):
    import numpy as np
    for d in ("a", "b"):
        line = run_bench_dump(tmp_path / d, "--utts", "8", "--steps", "3")
        assert line["steps"] == 3
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["loglik.npy", "loglik_rows.npy"] == sorted(os.listdir(tmp_path / "b"))
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 << 20
    ll, rows = np.load(tmp_path / "a" / "loglik.npy"), np.load(tmp_path / "a" / "loglik_rows.npy")
    assert ll.dtype == np.float32 and ll.shape[1] == 3000 and ll.shape[0] == rows.size < 8 * 998
    assert np.all(np.diff(rows) > 0) and rows[-1] < 8 * 998 and np.isfinite(ll).all()
    assert np.array_equal(rows, np.load(tmp_path / "b" / "loglik_rows.npy"))
    assert np.array_equal(ll, np.load(tmp_path / "b" / "loglik.npy"))


def test_flops_per_frame_matches_survey():
    sys.path.insert(0, ROOT)
    import bench
    assert bench.flops_per_frame(bench.CONFIGS["3"]) == 17530880   # SURVEY.md 8d
    assert bench.flops_per_frame(bench.CONFIGS["4"]) == 84901888
