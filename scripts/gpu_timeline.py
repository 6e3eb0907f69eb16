"""Where the 180 us of an env step go on the GPU's own clock (library built with -DFW_TIMELINE, FWGYM_LIB=...): first
block start / last block end of the init, attempt and env kernels, with the env kernel overlapped, or serial with
--serial (per-kernel profiling on: its event between the two kernels serialises them)."""
import ctypes, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import bench
from fwgym_b200 import FixedWingVecEnv, _capi
from fwgym_b200.config import DEFAULT_ENV_CONFIG
n = 65536
SERIAL = "--serial" in sys.argv[1:]
vec = FixedWingVecEnv(DEFAULT_ENV_CONFIG, n, config_kw=bench.CONFIG_KW, sim_config_kw=bench.SIM_KW, seed=1)
vec.reset()
lib = vec._lib
BURN = int(os.environ.get("FWGYM_TIMELINE_BURN", "0"))      # 200: the stationary episode mix of bench.py (auto-resets every step)
_b = torch.rand((16, n, 3), device="cuda") * 2 - 1
for i in range(BURN):
    vec.step_tensors(_b[i % 16])
acts = torch.rand((40, n, 3), device="cuda") * 2 - 1
flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
buf = (ctypes.c_ulonglong * 8)()
rows = []
vec.set_profiling(SERIAL)
for t in range(40):
    torch.cuda.synchronize()
    _capi.check(lib.fw_debug_timeline(None, 1))
    flush.zero_()          # like bench.py: the step is enqueued while the flush runs, so no host launch latency is exposed
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    vec.step_tensors(acts[t])
    e1.record()
    torch.cuda.synchronize()
    _capi.check(lib.fw_debug_timeline(buf, 0))
    b = np.array(list(buf), dtype=np.float64)
    if t >= 8:
        t0 = b[0]
        rows.append([(b[1] - t0), (b[2] - t0), (b[3] - t0), (b[4] - t0), (b[6] - t0), (b[5] - t0), b[7] / ((n + 127) // 128),
                     e0.elapsed_time(e1) * 1e6])
r = np.array(rows).mean(0) / 1e3
print("burn_in=%d overlap=%d  us from the first init block: init end %.1f | attempt start %.1f end %.1f | env first block resident %.1f, "
      "first past its wait %.1f, last end %.1f | mean env block run time %.1f | events around fw_step %.1f"
      % (BURN, 0 if SERIAL else 1, r[0], r[1], r[2], r[3], r[4], r[5], r[6], r[7]))
