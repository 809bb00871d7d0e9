"""bench.py's control flow against the engine as it is now, without a GPU (tests/_bench_dry.py): every config must come
out `exact`, every timed step must launch, and the line must carry the keys of the bench contract - at 1 rank and at 2 ranks
over gloo (weak + strong legs, halo exchange / all-gather / all-reduce inside timed loops, flush scripts replayed)."""
import json
import os
import socket
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


def _run(world, *args):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    procs = []
    for r in range(world):
        env = dict(os.environ)
        env.update({"RANK": str(r), "WORLD_SIZE": str(world), "LOCAL_RANK": str(r), "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": str(port),
                    "OMP_NUM_THREADS": "1"})
        procs.append(subprocess.Popen([sys.executable, os.path.join(HERE, "_bench_dry.py"), *args], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=280)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o[-3000:]
    return json.loads(outs[0].strip().splitlines()[-1])


@pytest.mark.timeout(300)
@pytest.mark.parametrize("world", [1, 2])
def test_bench_control_flow(world, tmp_path):
    d = _run(world, "--dump-outputs", str(tmp_path))
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
              "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks"):
        assert k in d, k
    assert d["n_gpus"] == world and d["exact"] is True and d["gpu_launches"] >= d["steps"]
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    for c in ("config3", "config4", "config5"):
        e = d["extra"][c]
        assert e["exact"] is True and e["roofline"]["launches_per_step"] >= 1, c
    if world > 1:
        assert d["strong"]["exact"] is True
        assert d["extra"]["config3"]["collectives_per_step"] >= 1 and d["extra"]["config5"]["collectives_per_step"] >= 1
        assert d["extra"]["config4"]["bytes_sent_per_rank_per_step"] > 0
    # --dump-outputs: B, C, D of the last timed step, whole at this size (200000 elements per rank)
    import numpy as onp

    assert sorted(os.listdir(tmp_path)) == ["B.npy", "C.npy", "D.npy"]
    B, C, D = (onp.load(tmp_path / (n + ".npy")) for n in "BCD")
    A = onp.arange(200000 * world) * 0.001  # (the engine's arange(N) / 1000.0, bit for bit)
    assert B.dtype == C.dtype == D.dtype == onp.float64 and D.shape == A.shape
    assert onp.allclose(B, onp.sin(A), rtol=1e-13, atol=1e-15) and onp.allclose(C, onp.cos(A), rtol=1e-13, atol=1e-15)
    assert onp.array_equal(D, B * B + C ** 2)


def test_dumped_sample_positions_do_not_depend_on_the_implementation(oracle_engine):
    """bench.host_sample draws the same blocks for an engine array as for the NumPy array it holds, within its byte budget,
    also when one slab along axis 0 is larger than the budget."""
    import numpy as onp

    sys.path.insert(0, os.path.join(HERE, ".."))
    import bench
    import ramba_b200 as rb

    x1 = onp.arange(100000) * 0.5
    x3 = (onp.arange(24 * 16 * 10) % 7).astype(onp.float32).reshape(24, 16, 10)
    for x, budget in [(x1, 8000), (x1, 8 * 100000), (x3, 4 * 16 * 10 * 3), (x3, 4 * 7)]:
        got = bench.host_sample(rb.fromarray(x), budget, onp.random.default_rng(0))
        exp = bench.host_sample(x, budget, onp.random.default_rng(0))
        assert got.dtype == x.dtype and got.nbytes <= budget and onp.array_equal(got, exp), (x.shape, budget)
    assert bench.host_sample(x1, 8000, onp.random.default_rng(0)).size < x1.size


def test_smoke_logic_on_the_oracle_backend(oracle_engine):
    """__graft_entry__.smoke() with the oracle backend standing in for cuda:0: its comparisons (chain vs the C restatement,
    Laplacian / affine sum / broadcast + axis sum bit-exact) must hold for the engine as it is now."""
    import inspect

    sys.path.insert(0, os.path.join(HERE, ".."))
    import __graft_entry__ as g

    src = inspect.getsource(g.smoke)
    assert "assert RT.launches > 0 and RT.is_cuda" in src
    src = src.replace("assert RT.launches > 0 and RT.is_cuda", "assert RT.launches > 0")
    ns = {}
    exec(src, dict(g.__dict__), ns)
    ns["smoke"]()
