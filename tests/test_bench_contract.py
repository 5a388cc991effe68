"""bench.py's host-side contract, checked without a GPU: the committed ncu capture belongs to the kernels in the tree (a capture
of other kernels would be reported as stale, not as traffic), the film digests the timed legs are checked against exist, the
CPU sample is a whole number of tiles per worker, and the reference arm prints the line the driver expects."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_ncu_capture_is_reported_only_for_the_kernels_it_was_taken_from(monkeypatch):
    """A capture whose stamp equals the hash of today's kernel sources is reported; any other capture yields None and says
    'stale' — so the line can never carry the traffic of kernels that are not the ones running."""
    with open(os.path.join(ROOT, "profiles", "r02", "traffic.json")) as f:
        stored = json.load(f)
    for key in ("c2", "c5"):
        monkeypatch.setattr(bench, "kernel_source_hash", lambda key=key: stored[key]["kernel_hash"])
        t = bench.ncu_traffic(key)
        assert t["traffic_state"] == "current" and t["traffic_commit"] == stored[key]["commit"]
        assert t["dram_bytes_per_launch"] > 0 and t["l2_bytes_per_launch"] > t["dram_bytes_per_launch"]
        monkeypatch.setattr(bench, "kernel_source_hash", lambda: "0" * 16)
        t = bench.ncu_traffic(key)
        assert t["traffic_state"].startswith("stale") and t["dram_bytes_per_launch"] is None and t["l2_bytes_per_launch"] is None


def test_kernel_source_hash_ignores_host_only_sources(tmp_path, monkeypatch):
    before = bench.kernel_source_hash()
    src = os.path.join(ROOT, "yuki_b200", "csrc")
    names = [n for n in os.listdir(src) if n.endswith(".cuh") or n in ("render.cu", "yk_libm.h", "yk_fastdiv.h")]
    assert "wf_trace.cuh" in names and "render.cu" in names and "multi.inl" not in names and "host_pbrt.cpp" not in names
    assert before == bench.kernel_source_hash() and len(before) == 16


def test_stored_film_digests_cover_the_timed_legs():
    with open(bench.DIGESTS) as f:
        stored = json.load(f)
    assert "c2_1024spp" in stored and bench.C5_DIGEST in stored
    assert bench.check_digest("c2_1024spp", stored["c2_1024spp"], False) == "ok"
    assert bench.check_digest("no_such_workload", "0" * 32, False) == "absent"
    try:
        bench.check_digest("c2_1024spp", "0" * 32, False)
    except SystemExit as e:
        assert "film digest" in str(e)
    else:
        raise AssertionError("a wrong film must stop the bench")


def test_reference_arm_prints_the_drivers_line():
    """`bench.py --impl reference` at 4 spp (a fraction of a second of CPU work): one JSON line on stdout with impl / cpu_baseline / e2e."""
    env = dict(os.environ)
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--spp-side", "2"],
                       capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, p.stdout
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["metric"] == "Msamples/s" and line["higher_is_better"] is True
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["value"] == line["value"] > 0
    assert line["e2e"] == {"value": line["value"], "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert np.isfinite(line["ms_per_step"])


def test_dump_outputs_fit_the_budget_and_sample_the_same_pixels_every_run(tmp_path):
    """--dump-outputs: the 1024x1024 film is written whole; a 3840x2160 film (--workload c5) is replaced by the same seeded pixel
    sample on every run, and one dump's files stay within the 64 MB budget."""
    counters = [3.5e9, 1e9, 2 ** 30, 5, 6, 7, 8]
    small = np.random.default_rng(1).random((1024, 1024, 3), dtype=np.float32)
    bench.dump_outputs(str(tmp_path / "small"), small, counters)
    assert np.array_equal(np.load(tmp_path / "small" / "film.npy"), small)
    got = np.load(tmp_path / "small" / "counters.npy")
    assert got.dtype == np.float64 and got.tolist() == counters
    big = np.random.default_rng(2).random((2160, 3840, 3), dtype=np.float32)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), big, counters)
        files = sorted(os.listdir(tmp_path / run))
        assert files == ["counters.npy", "film_sample.npy", "film_sample_index.npy"]
        assert sum(os.path.getsize(tmp_path / run / f) for f in files) <= bench.DUMP_LIMIT
    idx = np.load(tmp_path / "a" / "film_sample_index.npy")
    assert np.array_equal(idx, np.load(tmp_path / "b" / "film_sample_index.npy"))
    assert np.array_equal(np.load(tmp_path / "a" / "film_sample.npy"), big.reshape(-1, 3)[idx.astype(np.int64)])


def test_bench_refuses_zero_steps_and_a_reference_dump(tmp_path):
    for extra, msg in ((["--steps", "0"], "--steps must be at least 1"),
                       (["--impl", "reference", "--dump-outputs", str(tmp_path)], "the reference arm renders a sample of the tiles")):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, cwd=ROOT, timeout=600)
        assert p.returncode == 2 and msg in p.stderr, p.stderr
