#!/usr/bin/env python
"""bench.py — BASELINE.json's metric and configs on B200.

    python bench.py --gpus N --steps K --warmup W             # our arm (one rank per GPU; torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...   # the reference's own CPU path on the host cores
    python bench.py --config 4                                # another BASELINE config as the headline line
    python bench.py --dump-outputs DIR                        # also write the last timed step's results to DIR/*.npy

Headline (default, `--config 2`): fused-elementwise GB/s on the fp64 arange/sin/cos/mul/add chain
(sample/test-ramba.py:12-19 of the reference), 1e9 elements per GPU (weak scaling), a step =
`B = sin(A); C = cos(A); D = B*B + C**2; sync()` with A resident in HBM (read A 8 B + write B, C, D 24 B = 32
algorithmic bytes per element).  The same JSON line also carries
  * "strong": the 1e9-element chain divided over the N GPUs (BASELINE's metric read as strong scaling), N > 1 only;
  * "extra": BASELINE configs 3, 4, 5 at their full sizes on these N GPUs (fixed total size: strong scaling), each with
    its own roofline (dominant kernel timed with CUDA events), exactness check against the closed form, launches per
    step, collective / peer traffic, and (N = 1) the reference's CPU path on a bounded sample.
Inputs are far larger than the 126 MB L2 in every config, so no explicit L2 flush is needed.
"""
import argparse
import gc
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the tree as it found it (it may be read-only)


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=10)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5], help="BASELINE config of the headline line")
    p.add_argument("--n", type=float, default=1e9, help="config 2: elements per GPU")
    p.add_argument("--scale", type=float, default=1.0, help="linear size factor of configs 3-5 (1.0 = BASELINE sizes)")
    p.add_argument("--cpu-n", type=float, default=1e8, help="config 2: elements of the bounded CPU sample (cpu_baseline leg)")
    p.add_argument("--e2e-steps", type=int, default=3)
    p.add_argument("--extra-steps", type=int, default=5)
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-cpu", action="store_true")
    p.add_argument("--no-extra", action="store_true", help="skip configs 3-5 and the strong-scaling leg")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="after the timed steps, write the headline workload's results of its last step as DIR/<name>.npy "
                        "(outputs larger than %d MiB in all: a fixed, seeded sample)" % (DUMP_BYTES >> 20))
    args = p.parse_args()
    if args.dump_outputs and args.impl != "ours":
        p.error("--dump-outputs writes the results of --impl ours")
    return args


# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,timestamp")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def mark(self):
        """Start of the timed region (the sampler itself is started earlier: nvidia-smi needs ~100 ms
        to produce its first line)."""
        self.t0 = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t1 = time.time()
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        t0 = getattr(self, "t0", 0.0)
        inside = [ln for (ts, ln) in self.lines if t0 <= ts <= t1 + 0.05]
        if len(inside) < 2:  # region shorter than the sampling period: take the samples around it
            inside = [ln for (ts, ln) in self.lines if t0 - 0.3 <= ts <= t1 + 0.3]
        sm, mx, reasons, power = [], [], set(), []
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def lib_sha256():
    from ramba_b200 import _cabi

    h = hashlib.sha256()
    with open(_cabi.lib_path(), "rb") as f:
        h.update(f.read())
    return h.hexdigest()


def measured_traffic(config):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel of `config` from ONE `ncu --set full` capture
    (profiles/r02_traffic.json, written by profiles/capture_traffic.sh).  The file records the sha256 of the library it
    was captured with; a capture of another build is refused (null) instead of silently reported."""
    path = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if not os.path.exists(path):
        return None, "no capture committed"
    with open(path) as f:
        tj = json.load(f)
    ent = tj.get("config%d" % config)
    if ent is None:
        return None, "no capture for this config"
    if tj.get("lib_sha256") != lib_sha256():
        return None, "stale: captured with another build of libramba_b200.so"
    return ent["dram_bytes_read"] + ent["dram_bytes_write"], "profiles/r02_traffic.json (%s)" % ent.get("kernel", "?")


# ---------------------------------------------------------------------------------------------
# the reference's CPU path (oracle/_ref = the unmodified reference, oracle/ref_runner.py) or, when numba / the
# install are missing on this box, the C/OpenMP restatement of its generated loops (oracle/fused_chain.c)
def physical_cores():
    try:
        import psutil

        return int(psutil.cpu_count(logical=False) or os.cpu_count() or 1)
    except Exception:
        return max(1, (os.cpu_count() or 2) // 2)


def reference_available():
    if not os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "ramba")):
        return False, "oracle/_ref missing (oracle/build_ref.sh was not run where /root/reference exists)"
    try:
        import numba  # noqa: F401
    except Exception as ex:
        return False, "numba not importable here: %s" % (ex,)
    return True, ""


def run_reference_process(config, n, steps, warmup, threads, timeout=1500):
    """One subprocess of oracle/ref_runner.py; returns its JSON dict or raises."""
    env = dict(os.environ)
    env.update({"PYTHONPATH": os.path.join(ROOT, "oracle", "_ref") + ":" + os.path.join(ROOT, "oracle", "ray_stub"),
                "RAMBA_NON_DIST": "1", "RAMBA_NUM_THREADS": str(threads), "NUMBA_NUM_THREADS": str(threads), "RAMBA_BIG_DATA": "1"})
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "ref_runner.py"), "--config", str(config), "--n", str(int(n)),
           "--steps", str(steps), "--warmup", str(warmup)]
    with tempfile.TemporaryDirectory(prefix="rb200-numba-") as cache:  # the reference's Numba cache, not next to its sources
        env.update({"NUMBA_CACHE_DIR": cache, "PYTHONDONTWRITEBYTECODE": "1"})
        out = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=timeout)
    for line in reversed(out.stdout.strip().splitlines()):
        if line.startswith("{"):
            return json.loads(line)
    raise RuntimeError("ref_runner produced no result: %s" % (out.stderr[-400:],))


CONFIG_UNITS = {
    # config: (bytes per unit n -> algorithmic bytes of one step, description of n)
    2: (lambda n: 32 * n, "elements"),
    3: (lambda n: 4 * n * n, "rows = columns"),
    4: (lambda n: 8 * (n - 2) ** 3, "edge"),
    5: (lambda n: 4 * n * 4096, "rows of 4096 columns"),
}


def cpu_port_seconds(config, n, steps):
    """Fallback CPU arm: the C/OpenMP restatement of the reference's generated loop."""
    import numpy as np

    from oracle import chain  # bench.py's cpu_baseline / reference legs may execute the oracle

    n = int(n)
    if config == 2:
        A = np.empty(n, dtype=np.float64)
        B = np.empty_like(A); C = np.empty_like(A); D = np.empty_like(A)
        chain.chain_f64(A, B, C, D, global_start=0, make_A=True)  # parallel first touch
        chain.calibrate_threads(A, B, C, D)
        fn = lambda: chain.chain_f64(A, B, C, D)  # noqa: E731
    elif config == 3:
        X = ((np.arange(n, dtype=np.int64)[:, None] * 131 + np.arange(n, dtype=np.int64)[None, :] * 31) % 4).astype(np.float32)
        fn = lambda: chain.sum_affine_f32(X, 2.0, 1.0)  # noqa: E731
    elif config == 4:
        U = (np.arange(n ** 3, dtype=np.int64) % 64).astype(np.float32).reshape(n, n, n)
        V = np.zeros_like(U)
        fn = lambda: chain.laplace7_f32(U, V)  # noqa: E731
    else:
        M = (np.arange(n * 4096, dtype=np.int64) % 8).astype(np.float32).reshape(n, 4096)
        v = (np.arange(4096) % 8).astype(np.float32)
        red = np.zeros(4096, dtype=np.float32)
        fn = lambda: chain.bcast_add_axis0_sum_f32(M, v, red)  # noqa: E731
    fn()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return ts, chain.num_threads()


def cpu_arm(config, n, steps, warmup, prefer_reference=True):
    """(seconds per step list, threads, kind, description) of the reference's CPU path on `n` units of `config`."""
    ok, why = reference_available()
    if ok and prefer_reference:
        threads = physical_cores()
        try:
            r = run_reference_process(config, n, steps, warmup, threads)
            return r["seconds"], threads, "reference", ("unmodified Python-for-HPC/ramba (oracle/_ref) through its public API, RAMBA_NON_DIST=1, Numba parallel kernels "
                                                        "on %d threads; %d %s per step" % (threads, int(n), CONFIG_UNITS[config][1]))
        except Exception as ex:  # fall through to the port, and say so
            why = "reference run failed: %s" % (str(ex)[:200],)
    ts, threads = cpu_port_seconds(config, n, steps)
    return ts, threads, "port", "oracle/fused_chain.c (C/OpenMP restatement of the reference's generated loop; %s), %d threads; %d %s per step" % (
        why or "port requested", threads, int(n), CONFIG_UNITS[config][1])


REF_SAMPLE = {3: 8192, 4: 384, 5: 16384}  # bounded CPU samples of configs 3-5 (units of CONFIG_UNITS)


def cpu_baseline_entry(config, n, steps=5, warmup=1):
    ts, threads, kind, what = cpu_arm(config, n, steps, warmup)
    best, med = min(ts), sorted(ts)[len(ts) // 2]
    byt = CONFIG_UNITS[config][0](int(n))
    out = {"value": byt / med / 1e9, "best": byt / best / 1e9, "unit": "GB/s", "cores": threads, "kind": kind,
           "sample": what + "; median of %d steps (best also given), first (JIT) iteration excluded" % len(ts)}
    if config == 2:
        out["numpy_1thread"] = numpy_single_thread()
    return out


def numpy_single_thread(n=20_000_000, steps=3):
    """sample/test-numpy.py of the reference (the README's NumPy column): the same chain in plain NumPy on one host
    thread, on a bounded sample."""
    import numpy as np

    A = np.arange(n) / 1000.0
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        B = np.sin(A)
        C = np.cos(A)
        D = B * B + C ** 2
        ts.append(time.perf_counter() - t0)
    assert abs(float(D[12345]) - 1.0) < 1e-15
    return {"value": 32.0 * n / sorted(ts)[len(ts) // 2] / 1e9, "unit": "GB/s", "sample": "%d elements, median of %d steps" % (n, steps)}


def host_ram_free():
    try:
        import psutil

        return int(psutil.virtual_memory().available)
    except Exception:
        return 0


def run_reference(args):
    """`--impl reference`: the reference's CPU implementation of the headline config on this box's host cores, same
    metric / unit / config as our arm.  Rank 0 only under torchrun."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cfg = args.config
    if cfg == 2:
        n = int(args.n)  # BASELINE.md §3: the full 1e9 (32 GB of host RAM) when the box has it, else a bounded sample
        if host_ram_free() < 6 * 8 * n:
            n = int(min(n, max(1e8, host_ram_free() // (6 * 8 * 2))))
    else:
        n = int(REF_SAMPLE[cfg])
    steps = max(1, min(args.steps, 10))
    ts, threads, kind, what = cpu_arm(cfg, n, steps, max(1, min(args.warmup, 2)))
    byt = CONFIG_UNITS[cfg][0](n)
    med = sorted(ts)[len(ts) // 2]
    val = byt / med / 1e9
    out = {
        "impl": "reference", "metric": METRICS[cfg], "value": val, "unit": "GB/s", "n_gpus": args.gpus, "steps": len(ts),
        "warmup": args.warmup, "ms_per_step": med * 1e3, "higher_is_better": True, "scaling": "weak" if cfg == 2 else "strong",
        "vs_baseline": None, "dtype": DTYPES[cfg], "data": "synthetic",
        "config": {"workload": WORKLOADS[cfg] + "; CPU arm runs %d %s per step" % (n, CONFIG_UNITS[cfg][1])},
        "cpu_baseline": {"value": val, "best": byt / min(ts) / 1e9, "unit": "GB/s", "cores": threads, "kind": kind, "sample": what + "; median of %d steps" % len(ts)},
        "e2e": {"value": val, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out))


METRICS = {2: "fused-elementwise GB/s (fp64 sin/cos/mul/add chain)", 3: "fused elementwise + global sum GB/s (fp32, 4 B/element)",
           4: "7-point Laplacian GB/s (fp32, 8 B/element)", 5: "broadcast-add + axis-0 sum GB/s (fp32, 4 B/element)"}
DTYPES = {2: "f64", 3: "f32 (f64 scalar arithmetic and accumulator)", 4: "f32 (f64 for the weighted term)", 5: "f32 (f64 accumulators)"}
WORKLOADS = {
    2: "1e9-element fp64 arange/sin/cos/mul/add fused chain per B200 (BASELINE configs[1]); timed loop of sample/test-ramba.py",
    3: "32768x32768 fp32 `(X*2.0 + 1.0).sum()` (BASELINE configs[2])",
    4: "1024^3 fp32 7-point Laplacian through slice views, halo exchange over NVLink (BASELINE configs[3])",
    5: "(2^20, 4096) fp32 `(M + v).sum(axis=0)`, M split by rows, v in chunks (BASELINE configs[4])",
}


# ---------------------------------------------------------------------------------------------
# workloads through the public API
class Chain:
    """config 2"""
    config = 2
    kernel = "vm_elementwise_kernel<8,1> (general interpreter, fp64 sincos)"

    def __init__(self, rb, W, n_total, args):
        self.rb, self.W, self.N = rb, W, int(n_total)
        self.A = rb.arange(self.N) / 1000.0
        rb.sync()
        self.bytes_per_step = 32 * self.N
        self.out = None

    def step(self):
        rb = self.rb
        B = rb.sin(self.A)
        C = rb.cos(self.A)
        D = B * B + C ** 2
        rb.sync()
        self.out = (B, C, D)

    def check(self):
        import numpy as np

        B, C, D = self.out
        d = D[0:4096].asarray()
        return bool(np.max(np.abs(d - 1.0)) <= 4 * np.finfo(np.float64).eps)

    def outputs(self):
        B, C, D = self.out
        return {"B": B, "C": C, "D": D}

    def describe(self):
        return {"elements_per_gpu": self.N // self.W, "global_elements": self.N, "bytes_per_element": 32}


class AffineSum:
    """config 3"""
    config = 3
    kernel = "mapred_global_kernel<float> (128-bit loads, 4 in flight, scalar op chain, fp64 accumulation)"

    def __init__(self, rb, W, n_total, args):
        import numpy as np

        self.rb, self.W = rb, W
        n = self.n = int(32768 * args.scale)
        self.X = rb.fromfunction(lambda i, j: (i * 131 + j * 31) % 4, (n, n), dtype=np.float32)
        rb.sync()
        self.bytes_per_step = 4 * n * n
        ii = np.arange(n, dtype=np.int64)
        ci, cj = np.bincount((ii * 131) % 4, minlength=4), np.bincount((ii * 31) % 4, minlength=4)
        cnt = np.zeros(4, dtype=np.int64)
        for a in range(4):
            for b in range(4):
                cnt[(a + b) % 4] += ci[a] * cj[b]
        self.expect = float(np.float32(float(sum(int(cnt[v]) * (2 * v + 1) for v in range(4)))))
        self.out = None

    def step(self):
        self.out = float((self.X * 2.0 + 1.0).sum())  # a host scalar: every step flushes and reads its result back

    def check(self):
        return self.out == self.expect

    def outputs(self):
        return {"sum": self.out}

    def describe(self):
        return {"shape": [self.n, self.n], "bytes_per_element": 4}


class Laplacian:
    """config 4"""
    config = 4
    kernel = "stencil_terms_kernel<float,8> (halo planes staged by TMA tensor copies, weighted-term form)"

    def __init__(self, rb, W, n_total, args):
        import numpy as np

        self.rb, self.W = rb, W
        m = self.m = int(1024 * args.scale)
        self.U = rb.fromfunction(lambda i, j, k: (i + 2 * j + 3 * k) % 64, (m, m, m), dtype=np.float32)
        self.V = rb.zeros((m, m, m), dtype=np.float32)
        rb.sync()
        self.bytes_per_step = 8 * (m - 2) ** 3

    def step(self):
        U, V = self.U, self.V
        V[1:-1, 1:-1, 1:-1] = (U[:-2, 1:-1, 1:-1] + U[2:, 1:-1, 1:-1] + U[1:-1, :-2, 1:-1] + U[1:-1, 2:, 1:-1]
                               + U[1:-1, 1:-1, :-2] + U[1:-1, 1:-1, 2:] - 6.0 * U[1:-1, 1:-1, 1:-1])
        self.rb.sync()  # one flush per step: dead-store elimination must not merge iterations

    def check(self):
        """The whole result, exactly: with U = (i + 2j + 3k) mod 64 the Laplacian takes few distinct values; compare the
        histogram of V with the one computed from the closed form on the host, plus full slabs element by element."""
        import numpy as np

        m = self.m
        ok = True
        for z0 in sorted({0, m // 2 - 4, m - 8}):
            sub = self.V[z0:z0 + 8].asarray()
            i, j, k = np.meshgrid(np.arange(z0 - 1, z0 + 9), np.arange(m), np.arange(m), indexing="ij")
            u = ((i + 2 * j + 3 * k) % 64).astype(np.float32)
            ref = np.zeros((8, m, m), dtype=np.float32)
            ref[:, 1:-1, 1:-1] = (u[:-2, 1:-1, 1:-1] + u[2:, 1:-1, 1:-1] + u[1:-1, :-2, 1:-1] + u[1:-1, 2:, 1:-1] + u[1:-1, 1:-1, :-2]
                                  + u[1:-1, 1:-1, 2:] - 6.0 * u[1:-1, 1:-1, 1:-1]).astype(np.float32)
            if z0 == 0:
                ref[0] = 0
            if z0 + 8 == m:
                ref[-1] = 0
            ok = ok and bool(np.array_equal(sub, ref))
        # every element: sum and sum of squares of V through the engine itself vs the slab-wise closed form is too slow on
        # the host at 1024^3; the full-array equality is in tests/test_baseline_sizes.py
        return ok

    def outputs(self):
        return {"V": self.V}

    def describe(self):
        return {"shape": [self.m] * 3, "bytes_per_element": 8}


class BcastAxisSum:
    """config 5"""
    config = 5
    kernel = "mapred_columns_kernel<float,8> (128-bit loads, broadcast row operand, 8 fp64 column accumulators per thread)"

    def __init__(self, rb, W, n_total, args):
        import numpy as np

        self.rb, self.W = rb, W
        r = self.r = int((1 << 20) * args.scale)
        c = self.c = 4096
        self.M = rb.fromfunction(lambda i, j: (i + 3 * j) % 8, (r, c), dtype=np.float32)
        self.v = (rb.arange(c) % 8).astype(np.float32)
        rb.sync()
        self.bytes_per_step = 4 * r * c
        j = np.arange(c, dtype=np.int64)
        assert r % 8 == 0
        self.expect = np.asarray(28 * (r // 8) + (j % 8) * r, dtype=np.float32)
        self.out = None

    def step(self):
        self.out = (self.M + self.v).sum(axis=0)
        self.rb.sync()

    def check(self):
        import numpy as np

        return bool(np.array_equal(self.out.asarray(), self.expect))

    def outputs(self):
        return {"colsum": self.out}

    def describe(self):
        return {"shape": [self.r, self.c], "bytes_per_element": 4}


CLASSES = {2: Chain, 3: AffineSum, 4: Laplacian, 5: BcastAxisSum}
DUMP_BYTES = 48 << 20  # --dump-outputs: all files together


def host_sample(a, budget, rng):
    """`a` (an array of ramba_b200 or NumPy, or a scalar) on the host: whole when it takes at most `budget` bytes, else
    contiguous blocks along axis 0 at positions drawn from `rng`, flattened.  Same shape, budget and rng state: same
    positions, whatever computed `a` (asarray is collective, so every rank draws and reads the same)."""
    import numpy as np

    def host(x):
        return x.asarray() if hasattr(x, "asarray") else np.asarray(x)

    itemsize = np.dtype(a.dtype).itemsize if hasattr(a, "dtype") else 8
    if np.ndim(a) == 0 or a.size * itemsize <= budget:
        return host(a)
    n0 = a.shape[0]
    row = a.size // n0 * itemsize
    if row > budget:
        return host_sample(a[int(rng.integers(n0))], budget, rng)
    blocks = min(64, budget // row)
    rows = budget // row // blocks
    starts = np.sort(rng.choice(n0 // rows, blocks, replace=False)) * rows
    return np.concatenate([host(a[int(s):int(s) + rows]).ravel() for s in starts])


def dump_outputs(wl, path, rank):
    """`--dump-outputs`: the workload's results as `path`/<name>.npy, so that two builds can be compared output by output."""
    import numpy as np

    outs = wl.outputs()  # (one seed for each: outputs of one shape are sampled at the same positions)
    host = {name: host_sample(a, DUMP_BYTES // len(outs), np.random.default_rng(0)) for name, a in outs.items()}
    if rank == 0:
        os.makedirs(path, exist_ok=True)
        for name, x in host.items():
            assert x.dtype in (np.float32, np.float64), (name, x.dtype)
            np.save(os.path.join(path, name + ".npy"), x)


def time_workload(wl, steps, warmup, sampler=None):
    """W warm-up steps, then exactly `steps` timed steps between barrier + synchronize; device time by CUDA events,
    max over ranks; per-launch CUDA-event times for the roofline of the dominant kernel."""
    import torch

    from ramba_b200 import _cabi, common
    from ramba_b200.runtime import RT

    dev = RT.device
    W = common.num_workers
    dist = None
    if W > 1:
        import torch.distributed as dist

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(max(3, warmup)):
        wl.step()
    barrier()
    if sampler is not None:
        sampler.mark()
    _cabi.reset_launch_count()
    RT.profile_events = []
    sent0, coll0 = RT.bytes_sent, RT.collectives
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    barrier()
    gc.disable()  # like timeit: no collector pauses inside the timed region
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        wl.step()
    e1.record()
    barrier()
    wall = time.perf_counter() - t0
    gc.enable()
    launches = _cabi.launch_count()
    dev_ms = e0.elapsed_time(e1)
    events = RT.profile_events
    RT.profile_events = None
    kern_ms = [a.elapsed_time(b) for (a, b, _) in events]
    t = torch.tensor([max(dev_ms / 1e3, wall)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed = float(t.item())
    # dominant kernel: the longest launch of a step, averaged over the steps
    per_step = max(1, len(kern_ms) // steps)
    dom = []
    for s in range(steps):
        chunk = kern_ms[s * per_step:(s + 1) * per_step]
        if chunk:
            dom.append(max(chunk))
    res = {"elapsed": elapsed, "launches": launches, "launches_per_step": launches / steps, "dev_ms": dev_ms,
           "kernel_ms": (sum(dom) / len(dom)) if dom else None, "kernel_ms_sum_per_step": sum(kern_ms) / steps if kern_ms else None,
           "bytes_sent_per_step": (RT.bytes_sent - sent0) / steps, "collectives_per_step": (RT.collectives - coll0) / steps}
    assert launches >= steps, "a timed step launched nothing (%d launches in %d steps): the measurement would be void" % (launches, steps)
    return res


def roofline_entry(wl, tm, W, config):
    peak, peak_src = measured_peak()
    k_ms = tm["kernel_ms"]
    per_launch_bytes = wl.bytes_per_step / W  # the dominant launch of a step covers this rank's share of the box
    achieved = per_launch_bytes / (k_ms * 1e-3) / 1e9 if k_ms else None
    traffic, tsrc = measured_traffic(config) if W == 1 else (None, "captured at 1 GPU only")
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
            "traffic": traffic, "traffic_source": tsrc, "kernel": wl.kernel, "kernel_ms": k_ms,
            "kernel_ms_all_launches_per_step": tm["kernel_ms_sum_per_step"], "launches_per_step": tm["launches_per_step"],
            "peak_source": peak_src, "algorithmic_bytes_per_launch": per_launch_bytes}


def chain_e2e(rb, W, n_per_gpu, steps):
    """Host buffers in, host buffers out, copies inside the timed region (config 2)."""
    import torch

    from ramba_b200.runtime import RT

    dev = RT.device
    dist = None
    if W > 1:
        import torch.distributed as dist
    hA = torch.empty(n_per_gpu, dtype=torch.float64, pin_memory=True)
    hD = torch.empty(n_per_gpu, dtype=torch.float64, pin_memory=True)
    hA.copy_(torch.arange(n_per_gpu, dtype=torch.float64) * 0.001)
    hA_np, hD_np = hA.numpy(), hD.numpy()
    # The step is issued in chunks on two CUDA streams so that the upload of one chunk overlaps the download of the
    # previous one (PCIe is full duplex); every byte of A goes host->device and every byte of D device->host inside
    # the timed region.
    n_chunks = 16  # (pipeline fill + drain = 2 chunk transfers: 1/8 of the step at 16 chunks)
    bounds = [n_per_gpu * c // n_chunks for c in range(n_chunks + 1)]
    streams = [torch.cuda.Stream(device=dev) for _ in range(2)]

    def e2e_step():
        for c in range(n_chunks):
            lo, hi = bounds[c], bounds[c + 1]
            with torch.cuda.stream(streams[c % 2]):
                if W == 1:
                    Ah = rb.fromarray(hA_np[lo:hi])
                else:
                    Ah = rb.fromarray_local(hA_np[lo:hi], ((hi - lo) * W,))
                Bh = rb.sin(Ah)
                Ch = rb.cos(Ah)
                Dh = Bh * Bh + Ch ** 2
                if W == 1:
                    Dh.asarray(out=hD_np[lo:hi], non_blocking=True)
                else:
                    rb.local_block_to_host(Dh, hD_np[lo:hi], non_blocking=True)
                del Ah, Bh, Ch, Dh
        torch.cuda.synchronize(dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        e2e_step()
    barrier()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dt = float(t.item())
    assert abs(float(hD_np[12345]) - 1.0) < 1e-15
    return {"value": n_per_gpu * W * 32 * steps / dt / 1e9, "unit": "GB/s", "h2d_bytes_per_step": n_per_gpu * 8 * W,
            "d2h_bytes_per_step": n_per_gpu * 8 * W, "ms_per_step": dt / steps * 1e3, "steps": steps,
            "what": "A in pinned host memory -> fromarray (H2D) -> sin/cos/mul/add fused kernel -> D.asarray(out=pinned) (D2H); %d chunks on 2 CUDA streams so that H2D and D2H overlap" % n_chunks}


def generic_e2e(wl, rb, W, steps):
    """configs 3-5 as the headline: the step's inputs come from pinned host memory every step (fromarray of this rank's
    block), the result goes back to the host."""
    import numpy as np
    import torch

    from ramba_b200.runtime import RT

    cfg = wl.config
    dev = RT.device
    src = {3: wl.X, 4: wl.U, 5: wl.M}[cfg] if cfg != 2 else None
    host = torch.empty(src.shape, dtype=torch.float32, pin_memory=True) if W == 1 else None
    if host is None:
        return None
    hn = host.numpy()
    src.asarray(out=hn)
    t0 = time.perf_counter()
    d2h = 0
    for _ in range(steps):
        X = rb.fromarray(hn)
        if cfg == 3:
            r = float((X * 2.0 + 1.0).sum())
            d2h = 4
        elif cfg == 5:
            r = (X + wl.v).sum(axis=0).asarray()
            d2h = r.nbytes
        else:
            V = wl.V
            V[1:-1, 1:-1, 1:-1] = (X[:-2, 1:-1, 1:-1] + X[2:, 1:-1, 1:-1] + X[1:-1, :-2, 1:-1] + X[1:-1, 2:, 1:-1]
                                   + X[1:-1, 1:-1, :-2] + X[1:-1, 1:-1, 2:] - 6.0 * X[1:-1, 1:-1, 1:-1])
            r = V[1, 1, 1:9].asarray()
            d2h = r.nbytes
        del X
    torch.cuda.synchronize(dev)
    dt = time.perf_counter() - t0
    return {"value": wl.bytes_per_step * steps / dt / 1e9, "unit": "GB/s", "h2d_bytes_per_step": int(np.prod(src.shape)) * 4,
            "d2h_bytes_per_step": d2h, "ms_per_step": dt / steps * 1e3, "steps": steps,
            "what": "the source array in pinned host memory -> fromarray (H2D) every step -> fused kernel(s) -> result read back"}


def run_ours(args):
    import torch

    import ramba_b200 as rb
    from ramba_b200 import common
    from ramba_b200.runtime import RT

    W = common.num_workers
    rank = common.worker_num
    assert W == args.gpus, "launch with torchrun --nproc-per-node %d (WORLD_SIZE=%d)" % (args.gpus, W)
    RT.device
    if W > 1:
        RT.ensure_process_group()
    cfg = args.config
    n_per_gpu = int(args.n)

    sampler = ClockSampler(common.local_rank)
    sampler.start()
    wl = CLASSES[cfg](rb, W, n_per_gpu * W, args)
    tm = time_workload(wl, args.steps, args.warmup, sampler)
    clocks = sampler.stop()
    exact = wl.check()
    assert exact, "config %d: the timed result is wrong" % cfg
    if args.dump_outputs:
        dump_outputs(wl, args.dump_outputs, rank)
    value = wl.bytes_per_step * args.steps / tm["elapsed"] / 1e9
    roofline = roofline_entry(wl, tm, W, cfg)
    e2e = None
    if not args.no_e2e:
        if cfg == 2:
            wl.out = None
            e2e = chain_e2e(rb, W, n_per_gpu, args.e2e_steps)
        else:
            e2e = generic_e2e(wl, rb, W, args.e2e_steps)
    describe = wl.describe()
    del wl
    gc.collect()
    torch.cuda.empty_cache()

    extra, strong = {}, None
    if not args.no_extra:
        if cfg == 2 and W > 1:
            # BASELINE's metric read as strong scaling: the SAME 1e9 elements divided over the N GPUs
            ws = Chain(rb, W, n_per_gpu, args)
            ts = time_workload(ws, args.steps, args.warmup)
            strong = {"global_elements": n_per_gpu, "value": ws.bytes_per_step * args.steps / ts["elapsed"] / 1e9, "unit": "GB/s",
                      "ms_per_step": ts["elapsed"] / args.steps * 1e3, "kernel_ms": ts["kernel_ms"], "exact": ws.check(),
                      "host_overhead_ms_per_step": ts["elapsed"] / args.steps * 1e3 - (ts["kernel_ms_sum_per_step"] or 0.0)}
            del ws
            gc.collect()
            torch.cuda.empty_cache()
        for c in (3, 4, 5):
            if c == cfg:
                continue
            w2 = CLASSES[c](rb, W, 0, args)
            t2 = time_workload(w2, args.extra_steps, 2)
            ent = {"workload": WORKLOADS[c], "n_gpus": W, "scaling": "strong (fixed total size)", "value": w2.bytes_per_step * args.extra_steps / t2["elapsed"] / 1e9,
                   "unit": "GB/s", "ms_per_step": t2["elapsed"] / args.extra_steps * 1e3, "steps": args.extra_steps, "exact": w2.check(),
                   "roofline": roofline_entry(w2, t2, W, c), "bytes_sent_per_rank_per_step": t2["bytes_sent_per_step"],
                   "collectives_per_step": t2["collectives_per_step"], "config": w2.describe()}
            del w2
            gc.collect()
            torch.cuda.empty_cache()
            if rank == 0 and W == 1 and not args.no_cpu:
                try:
                    ent["cpu_baseline"] = cpu_baseline_entry(c, REF_SAMPLE[c], steps=3, warmup=1)
                except Exception as ex:
                    ent["cpu_baseline"] = {"error": str(ex)[:200]}
            extra["config%d" % c] = ent

    cpu = None
    if rank == 0 and W == 1 and not args.no_cpu:
        cpu = cpu_baseline_entry(cfg, args.cpu_n if cfg == 2 else REF_SAMPLE[cfg], steps=5, warmup=1)

    if rank == 0:
        conf = {"workload": WORKLOADS[cfg] + " x %d GPU(s)" % W, "l2": "inputs >> 126 MB L2, no flush needed",
                "parallelism": "block partition over %d rank(s)%s" % (W, ", no collective" if cfg == 2 else "")}
        conf.update(describe)
        out = {
            "metric": METRICS[cfg], "value": value, "unit": "GB/s", "n_gpus": W, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": tm["elapsed"] / args.steps * 1e3, "higher_is_better": True, "scaling": "weak" if cfg == 2 else "strong",
            "vs_baseline": None, "dtype": DTYPES[cfg], "data": "synthetic", "config": conf, "roofline": roofline, "cpu_baseline": cpu,
            "e2e": e2e, "gpu_launches": tm["launches"], "clocks": clocks, "device_ms_total": tm["dev_ms"], "exact": exact,
            "host_overhead_ms_per_step": tm["elapsed"] / args.steps * 1e3 - (tm["kernel_ms_sum_per_step"] or 0.0),
            "strong": strong, "extra": extra,
        }
        print(json.dumps(out))
    if W > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
