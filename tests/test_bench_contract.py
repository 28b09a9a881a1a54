"""bench.py's reference arm runs on the host alone (no GPU, no copy of the reference project) and prints one JSON line
with the result keys; the N>1 launch lets rank 0 print and the other ranks exit 0 without work. --dump-outputs writes
the result arrays of the last timed step, the same from run to run."""
import json
import os
import subprocess
import sys
import types

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None):
    env = dict(os.environ)
    env.pop("RANK", None); env.pop("WORLD_SIZE", None); env.pop("LOCAL_RANK", None)
    env["CUDA_VISIBLE_DEVICES"] = ""
    if extra_env:
        env.update(extra_env)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tiny",
                           "--steps", "1", "--warmup", "0"], capture_output=True, text=True, env=env, timeout=600)


def test_reference_arm_prints_the_contract_line():
    r = _run()
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    assert d["metric"] == "keymask_discovery_frames_per_sec" and d["unit"] == "frames/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("tiny")


def test_reference_arm_other_ranks_exit_without_work():
    r = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0, r.stderr[-2000:]
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]


def test_reference_arm_ignores_torchrun_thread_cap():
    """torchrun exports OMP_NUM_THREADS=1 to its workers; the CPU arm must still use every host core, or the per-N
    ratios of the scaling run are not comparable (round-1 verdict)."""
    r = _run({"OMP_NUM_THREADS": "1", "RANK": "0", "WORLD_SIZE": "2", "LOCAL_RANK": "0"})
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
    assert d["cpu_baseline"]["cores"] == len(os.sched_getaffinity(0))
    # both arms print the same `config` (bench.make_config)
    assert set(d["config"]) == {"workload", "videos_per_gpu", "frames_per_video", "resolution", "masks_per_frame",
                                "tracks_per_query", "queries_per_video", "point_order", "partition", "cache"}


def test_reference_arm_of_a_list_workload():
    """--impl reference --workload c4: the CPU port on one query of a few videos of the list (down-scaled here), same
    contract line, strong scaling."""
    env = dict(os.environ)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        env.pop(k, None)
    env["CUDA_VISIBLE_DEVICES"] = ""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c4", "--list-videos", "4",
                        "--list-scale", "0.1", "--steps", "1", "--warmup", "0"], capture_output=True, text=True, env=env, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
    assert d["impl"] == "reference" and d["scaling"] == "strong" and d["value"] > 0
    assert d["config"]["workload"].startswith("c4") and d["cpu_baseline"]["kind"] == "port"
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]


def _fake_batch(T=5, L=4, Nms=(7, 3)):
    """the attributes of a Batch that bench.dump_outputs reads, on the host; video 1 failed stage B"""
    rng = np.random.default_rng(1)
    R = sum(Nms)
    ri = np.stack([rng.integers(0, 2, R), rng.integers(-1, 2, R), rng.integers(0, 2, R), rng.integers(2, T, R)], 1).astype(np.int32)
    vidinfo = np.zeros((len(Nms), 8), np.int32)
    vidinfo[0, 1] = 1
    summ = dict(vidinfo=vidinfo, clusterinfo=np.zeros((len(Nms), 16, 16), np.int32), rowinfo=ri,
                glabel=np.arange(R, dtype=np.int32), one2x=np.zeros(R, np.int32))
    i32 = lambda n: torch.arange(n, dtype=torch.int32)
    return types.SimpleNamespace(host_descs=[types.SimpleNamespace(T=T, L=L, Nm=n) for n in Nms], device=torch.device("cpu"),
                                 fetch_summary=lambda: summ, qframe=i32(R), qlabel=i32(R), labels1=i32(R),
                                 V=torch.rand(R * T), mbits=torch.tensor([-1, 5, 7], dtype=torch.int32),
                                 hits=i32(R * T * L), uniq=i32(R * T))


@pytest.mark.parametrize("budget", [60_000_000, 3000])
def test_dump_outputs_holds_the_voted_tiles_within_the_budget(budget, tmp_path):
    """--dump-outputs on the host side: float32 / float64 files only, no more bytes than the budget, a fixed sample where
    an array does not fit, and `votes` holds exactly the tiles of candidate rows of videos that passed stage B."""
    import bench
    b = _fake_batch()
    runs = []
    for k in range(2):
        d = tmp_path / str(k)
        bench.dump_outputs(str(d), b, budget=budget)
        runs.append({f: np.load(d / f) for f in sorted(os.listdir(d))})
    assert list(runs[0]) == list(runs[1]) and all(np.array_equal(runs[0][f], runs[1][f]) for f in runs[0])
    files = runs[0]
    assert all(a.dtype in (np.float32, np.float64) for a in files.values())
    assert sum(a.nbytes for a in files.values()) <= budget
    assert ("clusterinfo_rows.npy" in files) == (budget < 4096)
    assert files["match_bits.npy"].tolist() == [2.0 ** 32 - 1, 5.0, 7.0]
    T, L = 5, 4
    ri = b.fetch_summary()["rowinfo"]
    want = [(r, f) for r in range(7) if ri[r, 1] >= 0 for f in range(ri[r, 2], ri[r, 3] + 1)]
    v = files["votes.npy"]
    assert [(int(r), int(f)) for r, f in v[:, :2]] == want
    for r, f, u, *h in v.tolist():
        t = int(r) * T + int(f)
        assert u == t and h == list(range(t * L, t * L + L))


def test_dump_list_results_keeps_every_field_and_digest(tmp_path):
    import bench
    res = [{"name": f"v{i}", "frames": 20 + i, "queries": 40 + i, "candidates": 30 + i, "status": 1 - 2 * (i % 2), "clusters": 2,
            "keymasks": 7 * i, "tiles": 100 + i, "digest": bytes(range(i, i + 32)).hex()} for i in range(3)]
    bench.dump_list_results(str(tmp_path), res)
    assert sorted(os.listdir(tmp_path)) == ["digests.npy", "videos.npy"]
    v, dg = np.load(tmp_path / "videos.npy"), np.load(tmp_path / "digests.npy")
    assert v.dtype == dg.dtype == np.float64
    assert v.tolist() == [[20 + i, 40 + i, 30 + i, 1 - 2 * (i % 2), 2, 7 * i, 100 + i] for i in range(3)]
    assert [bytes(int(x) for x in row).hex() for row in dg] == [r["digest"] for r in res]


def _bench_runs(tmp_path, args, steps):
    """bench.py with `args` once per entry of `steps`, each with --dump-outputs: [(JSON line, {file: array})]"""
    env = dict(os.environ)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        env.pop(k, None)
    out = []
    for k in steps:
        d = tmp_path / f"run{len(out)}"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args + ["--steps", str(k), "--dump-outputs", str(d)],
                           capture_output=True, text=True, env=env, timeout=900)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
        assert line["steps"] == k
        out.append((line, {f: np.load(d / f) for f in sorted(os.listdir(d))}))
    for _, files in out:
        assert list(files) == list(out[0][1]) and sum(a.nbytes for a in files.values()) <= 64 * 2 ** 20
        for f, a in files.items():
            assert a.dtype in (np.float32, np.float64) and np.array_equal(a, out[0][1][f], equal_nan=True), f
    return out


@pytest.mark.gpu
def test_batch_steps_and_dumped_outputs(tmp_path):
    """--steps K enqueues K steps in the timed region (launches in proportion), and the results of the last step are the
    same whatever K is."""
    (l2, files), (l3, _) = _bench_runs(tmp_path, ["--workload", "tiny", "--warmup", "3", "--no-e2e", "--no-cpu", "--no-k1"], [2, 3])
    assert l2["parity_check"] == l3["parity_check"] == "ok"
    assert l2["gpu_launches"] > 0 and 2 * l3["gpu_launches"] == 3 * l2["gpu_launches"]
    assert {"votes.npy", "V.npy", "rowinfo.npy", "match_bits.npy"} <= set(files) and len(files["votes.npy"]) > 0


@pytest.mark.gpu
def test_list_workload_steps_and_dumped_outputs(tmp_path):
    """c4 (a list workload): --steps K runs K timed passes over the list (launches, frames and K2 tiles in proportion), and
    the per-video results of the last pass - the ones the digest is computed from - are the same whatever K is."""
    (l1, files), (l2, _) = _bench_runs(tmp_path, ["--workload", "c4", "--list-videos", "4", "--list-scale", "0.1", "--no-cpu"], [1, 2])
    assert l1["results"]["digest"] == l2["results"]["digest"] and l1["results"]["videos_ok"] > 0
    assert l1["gpu_launches"] > 0 and l2["gpu_launches"] == 2 * l1["gpu_launches"]
    assert l2["roofline"]["tiles"] == 2 * l1["roofline"]["tiles"] > 0
    v, dg = files["videos.npy"], files["digests.npy"]
    assert v.shape == (4, 7) and dg.shape == (4, 32) and v[:, 0].sum() == l1["config"]["frames"]
    assert int((v[:, 3] == 1).sum()) == l1["results"]["videos_ok"] and int(v[:, 5].sum()) == l1["results"]["keymasks"]
