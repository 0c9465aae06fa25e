"""bench.py contract checks that need no GPU: the reference arm (CPU oracle port) prints ONE
JSON line with the agreed keys, non-zero ranks stay silent, and the own arm refuses to run
without a CUDA device instead of falling back to anything."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = ["--steps", "2", "--warmup", "1", "--batch", "8", "--layers", "1", "--hidden", "16"]


def run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, cwd=ROOT,
                          env=e, capture_output=True, text=True, timeout=600)


def test_reference_arm_prints_one_json_line():
    r = run(["--impl", "reference", "--gpus", "1"] + SMALL)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "graphs/s" and d["higher_is_better"] is True
    assert d["metric"] == "sswl_plus_zinc_shape_train_graphs_per_s" and d["value"] > 0
    assert d["vs_baseline"] is None and d["scaling"] == "strong" and d["data"] == "synthetic"
    assert d["steps"] == 2 and d["warmup"] == 1 and d["config"]["global_batch"] == 8
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_exit_silently():
    r = run(["--impl", "reference", "--gpus", "2"] + SMALL, {"RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_own_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    r = run(["--gpus", "1", "--steps", "1", "--warmup", "1"])
    assert r.returncode != 0
    assert "no CPU path" in (r.stderr + r.stdout)


def test_steps_below_one_are_refused():
    r = run(["--impl", "reference", "--steps", "0"])
    assert r.returncode != 0 and "--steps must be at least 1" in r.stderr


def test_dump_outputs_writes_float_arrays_within_the_budget(tmp_path):
    """--dump-outputs: every array as <name>.npy in float32 (float64 kept); above the byte budget
    the same seeded sample of positions in every run."""
    import importlib.util
    import numpy as np
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    rng = np.random.default_rng(1)
    arrays = {"loss": np.float32([0.5]), "pred": rng.standard_normal((50, 1)).astype(np.float32),
              "param.w": rng.standard_normal((300, 200)), "count": np.arange(7)}
    b.dump_outputs(str(tmp_path / "all"), arrays)
    for k, v in arrays.items():
        got = np.load(tmp_path / "all" / f"{k}.npy")
        assert got.dtype == (np.float64 if v.dtype == np.float64 else np.float32), k
        assert np.array_equal(got, v), k
    budget = 100_000
    for d in ("a", "b"):
        b.dump_outputs(str(tmp_path / d), arrays, budget=budget)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(f"{k}.npy" for k in arrays)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= budget
    for f in files:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)), f
    w = np.load(tmp_path / "a" / "param.w.npy")
    assert 0 < w.size < arrays["param.w"].size and np.isin(w, arrays["param.w"]).all()


def test_reference_arm_other_workloads():
    """The dense PPGN and the sr25 DSSGNN / I2 arms run on the CPU oracle too."""
    for wl in ("ppgn_dd", "dssgnn_sr25", "i2_sr25"):
        r = run(["--impl", "reference", "--workload", wl, "--steps", "1", "--warmup", "1",
                 "--ref-batch", "2", "--batch", "2", "--layers", "1", "--hidden", "8"])
        assert r.returncode == 0, r.stderr[-2000:]
        d = json.loads(r.stdout.strip().splitlines()[-1])
        assert d["value"] > 0 and d["config"]["global_batch"] == 2 and wl.split("_")[0] in d["metric"]


def test_strong_scaling_shards_cover_the_global_batch_and_are_balanced():
    """bench.py --gpus N (strong scaling): the ranks' shards are a disjoint cover of the 1-GPU
    job's global batch, equal in graph count and within 3 % in tuple count."""
    import importlib.util
    import numpy as np
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    argv, sys.argv = sys.argv, ["bench.py"]
    try:
        spec.loader.exec_module(b)
        args = b.parse()
    finally:
        sys.argv = argv
    world, per = 4, 12
    shards = [b.host_batches(args, per, r, 1, world)[0] for r in range(world)]
    whole = b.host_batches(args, per * world, 0, 1, 1)
    from pygho_b200.hodata.synthetic import make_batch
    ref = make_batch(per * world, seed=0)
    assert sum(s.num_graphs for s in shards) == ref.num_graphs
    assert sum(s.num_nodes for s in shards) == ref.num_nodes
    assert sum(s.tupleid.shape[1] for s in shards) == ref.tupleid.shape[1]
    assert sorted(np.concatenate([s.y for s in shards]).tolist()) == sorted(ref.y.tolist())
    t = [s.tupleid.shape[1] for s in shards]
    assert all(s.num_graphs == per for s in shards) and max(t) <= 1.03 * min(t), t
    assert whole[0].num_graphs == per * world
