"""bench.py without a GPU: the algorithmic-byte formulas the roofline fractions divide by (SURVEY §8d, DESIGN §4) and
the JSON line of the reference arm (the one leg of bench.py that runs on host cores only)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_algorithmic_bytes_of_the_headline_workload():
    import bench

    n, e, k, f = 89250, 899756, 256, 500
    assert bench.bytes_bfs(n, e, k) == 4 * (4 * (n + 1) + 4 * e + 8 * e + 16 * n) + 2 * n * k == 96_024_304
    assert bench.bytes_epilogue(n, k, f) == 137_088_000 + 357_000_000
    assert bench.bytes_bfs(n, e, 1) == bench.bytes_bfs(n, e, 64) - 2 * n * 63  # one lane word up to 64 anchors
    assert bench.bytes_csr(n, e, e) == 32 * e + 8 * e + 28 * n
    cfg = bench.headline_config(__import__("graphpope_b200.synth", fromlist=["SHAPES"]).SHAPES["flickr-shape"], 4, e)
    assert cfg["total_anchors"] == 1024 and "256 anchors per GPU" in cfg["workload"] and "model" not in cfg


def test_reference_arm_prints_the_contract_line():
    env = dict(os.environ, GP_BENCH_REF_BUDGET_S="3", CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["metric"] and line["unit"] == line["cpu_baseline"]["unit"]
    assert line["higher_is_better"] is True and line["vs_baseline"] is None and line["n_gpus"] == 1
    assert line["value"] > 0 and line["value"] == line["cpu_baseline"]["value"] == line["e2e"]["value"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert "workload" in line["config"] and line["steps"] == 1 and line["warmup"] == 0
    # a non-zero rank of a torchrun launch prints nothing and exits 0
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT,
                       env=dict(env, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1"))
    assert r.returncode == 0 and not [ln for ln in r.stdout.splitlines() if ln.startswith("{")]


def test_a_failing_secondary_line_is_reported_not_fatal(capsys):
    import bench

    def boom(x):
        raise RuntimeError("CUDA out of memory (simulated) %d" % x)

    res, ok = bench.guarded(boom, 7)
    assert ok is False and res["parity_checked"] is False and "simulated) 7" in res["error"]
    assert bench.guarded(lambda a, b: ({"v": a + b}, True), 1, 2) == ({"v": 3}, True)


def test_dump_outputs_row_sample_and_argument_checks():
    import bench

    rows = bench.dump_rows(89250, 756)  # headline matrix, 270 MB: a fixed row sample under 64 MB
    assert 4 * 756 * rows.size <= bench.DUMP_BYTES < 64_000_000 and rows.size > 19_000
    assert np.all(np.diff(rows) > 0) and rows[-1] < 89250
    assert np.array_equal(rows, bench.dump_rows(89250, 756))
    assert np.array_equal(bench.dump_rows(1000, 756), np.arange(1000))
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True,
                           timeout=300, env=env, cwd=ROOT)
        assert r.returncode == 2 and "error:" in r.stderr, extra


@pytest.mark.gpu
def test_dump_outputs_holds_the_last_timed_step(tmp_path):
    """bench.py --dump-outputs: the row sample of the headline [N, F+K] matrix, x in columns [0, F) and the features
    bit-equal to the C oracle."""
    import torch

    import bench
    from graphpope_b200 import synth
    from oracle import cbfs

    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1",
                        "--no-cpu-baseline", "--no-secondary", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])["steps"] == 2
    assert sorted(os.listdir(tmp_path)) == ["features.npy"]
    got = np.load(tmp_path / "features.npy")
    shape = synth.FLICKR_SHAPE
    n, f = shape.num_nodes, shape.num_features
    rows = bench.dump_rows(n, f + bench.K_PER_GPU)
    assert got.dtype == np.float32 and got.shape == (rows.size, f + bench.K_PER_GPU)
    assert os.path.getsize(tmp_path / "features.npy") <= 64_000_000
    x = torch.randn(n, f, device="cuda", generator=torch.Generator("cuda").manual_seed(1)).cpu().numpy()
    assert np.array_equal(got[:, :f], x[rows])
    ei = synth.make_graph(shape)
    anchors = synth.stochastic_anchors(n, bench.K_PER_GPU, 42)
    want = cbfs.normalise(cbfs.bfs_hops(cbfs.InCsr(ei, n), anchors))[rows]
    assert np.array_equal(got[:, f:].view(np.uint32), want.view(np.uint32))
