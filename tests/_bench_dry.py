"""TEST-ONLY: dry run of bench.py's own arm without a GPU - the oracle backend stands in for the CUDA library and a
minimal fake of the torch.cuda calls bench.py makes (events, streams, synchronize, pinned memory) for the device, so that
the script's control flow (warm-up, timed loop, per-launch events, exactness checks, e2e leg with two streams, strong leg,
extra configs, the JSON line) runs against the engine as it is NOW.  The numbers it prints mean nothing."""
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, ".."))
sys.path.insert(0, HERE)
import torch  # noqa: E402

import _oracle_backend  # noqa: E402

_oracle_backend.install()

class Ev:
    def __init__(self, enable_timing=True): self.t = None
    def record(self, *a): self.t = time.perf_counter()
    def elapsed_time(self, other): return (other.t - self.t) * 1e3
    def synchronize(self): pass
class St:
    def __init__(self, device=None): pass
    cuda_stream = 0
class ctx:
    def __init__(self, s): pass
    def __enter__(self): return self
    def __exit__(self, *a): return False
torch.cuda.Event = Ev
torch.cuda.Stream = St
torch.cuda.stream = ctx
torch.cuda.synchronize = lambda *a, **k: None
torch.cuda.empty_cache = lambda: None
torch.cuda.is_available = lambda: True
torch.cuda.mem_get_info = lambda *a: (100 << 30, 180 << 30)
torch.cuda.get_device_name = lambda *a: "fake"
_empty = torch.empty
def empty(*a, **k):
    k.pop("pin_memory", None)
    return _empty(*a, **k)
torch.empty = empty
from ramba_b200.runtime import RT
be = RT.backend
be.timing = True
be.events = lambda: (Ev(), Ev())
from ramba_b200 import _cabi
cnt = [0]
orig_run = be.run
def run(fop, stream=None):
    cnt[0] += 1
    return orig_run(fop, stream)
be.run = run
_cabi.launch_count = lambda: cnt[0]
_cabi.reset_launch_count = lambda: cnt.__setitem__(0, 0)
import bench
sys.argv = ["bench.py", "--gpus", os.environ.get("WORLD_SIZE", "1"), "--steps", "3", "--warmup", "3", "--n", "200000", "--scale", "0.03125", "--no-cpu",
            "--extra-steps", "2", "--e2e-steps", "2"] + sys.argv[1:]
bench.main()
