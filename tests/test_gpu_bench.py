"""bench.py as a user runs it: --steps sets the number of timed steps of every workload, and --dump-outputs writes
what the last timed step returned -- for the sweep, bit for bit the weights the CPU oracle holds after the same
number of steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIGHT = ["--no-sweep", "--no-secondary", "--no-cpu-baseline", "--no-e2e", "--no-parity"]


def run_bench(*args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + [str(a) for a in args] + LIGHT,
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["sweep", "resnet50", "bert", "rsp", "resnet50-train", "bert-train"])
def test_steps_sets_the_timed_steps_and_outputs_are_dumped(workload, tmp_path):
    line = run_bench("--workload", workload, "--steps", 7, "--warmup", 1, "--dump-outputs", tmp_path)
    assert line["steps"] == 7
    files = sorted(os.listdir(tmp_path))
    assert files and all(f.endswith(".npy") for f in files), files
    assert sum(os.path.getsize(tmp_path / f) for f in files) <= 64 << 20
    for f in files:
        a = np.load(tmp_path / f)
        assert a.dtype in (np.float32, np.float64) and a.size > 0 and np.all(np.isfinite(a)), f


@pytest.mark.gpu
def test_dumped_sweep_outputs_are_the_last_timed_step(tmp_path):
    import bench
    from oracle import oracle as O
    steps, warmup = 6, 4
    run_bench("--steps", steps, "--warmup", warmup, "--dump-outputs", tmp_path)
    shapes = bench.keyset("sweep")
    keys = list(range(len(shapes)))
    _, kw, oname, _ = bench.OPTIMIZERS["sgd"]
    grads = bench.rank_grads(0, shapes)
    okv = O.OracleKVStore("device")
    okv.init(keys, bench.initial_weights(shapes))
    okv.set_optimizer(O.OracleOptimizer(oname, **kw))
    for _ in range(max(3, warmup) + steps):          # bench.py's untimed warm-up steps, then the timed ones
        okv.push(keys, [[grads[k]] for k in keys])
    for k, (s, c) in enumerate(zip(shapes, bench.dump_counts([bench.nelem(s) for s in shapes]))):
        want = np.empty(s, np.float32)
        okv.pull(k, want)
        if c < want.size:
            want = want.reshape(-1)[np.sort(np.random.default_rng(k).choice(want.size, c, replace=False))]
        got = np.load(tmp_path / ("out_%03d.npy" % k))
        assert got.shape == want.shape and np.array_equal(got.view(np.uint32), want.view(np.uint32)), k
