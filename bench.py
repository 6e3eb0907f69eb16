#!/usr/bin/env python
"""Headline benchmark: env-steps/s of the batched FixedWingAircraft.step hot path (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W            # this framework (CUDA kernels), one rank per GPU
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port) on host cores

Workload (config.workload): BASELINE.json configs[2] — 65536 envs per GPU, Dryden turbulence (moderate) + observation
noise, fp64 dopri5 — weak scaling over GPUs, no collective on the step path (NCCL only all-reduces the episode
metric sums and the timing).  A "step" is one VecEnv.step of every env of the rank (dynamics kernel + env kernel).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ENVS_PER_GPU = 65536
WORKLOAD = "65536 envs/GPU, fixed_wing_config.json, Dryden turbulence moderate + obs noise std 0.1, fp64 dopri5 (BASELINE configs[2])"
CONFIG_KW = {"observation": {"noise": {"mean": 0, "var": 0.1}}}
SIM_KW = {"turbulence": True, "turbulence_intensity": "moderate"}
# algorithmic work per env step (SURVEY §8d): F = 1080 + 3660 * k flops, k = dopri5 attempts (counted on device)
F_FIXED, F_ATTEMPT = 1080.0, 3660.0
ENV_BYTES_PER_STEP = 480.0   # env kernel algorithmic bytes per env step (SURVEY §8d)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="fwgym", choices=["fwgym", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=ENVS_PER_GPU)
    ap.add_argument("--burn-in", type=int, default=200,
                    help="untimed env steps after the reset, before the warm-up: every env starts its first episode at the "
                         "same moment, and with random actions the whole batch reaches stall / failure together around "
                         "step 50-65 (a burst of dopri5 stragglers with 15-35 attempts); after ~200 steps the episode ages "
                         "are mixed and the step time is the stationary one")
    ap.add_argument("--cpu-baseline-seconds", type=float, default=20.0)
    ap.add_argument("--e2e-steps", type=int, default=0,
                    help="steps of the end-to-end passes (default: --steps; a 20-step window is 4-8 ms of wall clock and "
                         "+-10 %% noisy, 200 steps give a steadier e2e figure)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned to rank 0's caller (obs, reward, "
                         "done, term) as DIR/<name>.npy; the inputs depend only on the arguments, so two builds can be "
                         "compared output for output")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "fwgym":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl fwgym)")
    return a


DUMP_LIMIT_BYTES = 60 * 1024 * 1024     # keeps a dump, .npy headers included, under 64 MB


def dump_outputs(path, arrays, limit=DUMP_LIMIT_BYTES):
    """Write the per-env host arrays of `arrays` (name -> [N, ...], float32 or float64) as path/<name>.npy.  Above
    `limit` bytes in all, every array keeps the same fixed, seeded sample of env rows, ascending, and env_index.npy
    (float64) lists them."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    n = len(next(iter(arrays.values())))
    row_bytes = sum(x[:1].nbytes for x in arrays.values())
    if n * row_bytes > limit:
        keep = limit // (row_bytes + 8)     # + the float64 index entry of each kept row
        idx = np.sort(np.random.RandomState(0).choice(n, keep, replace=False))
        arrays = {k: x[idx] for k, x in arrays.items()}
        arrays["env_index"] = idx.astype(np.float64)
    for k, x in arrays.items():
        np.save(os.path.join(path, k + ".npy"), x)


# ------------------------------------------------------------------------------------------------ CPU reference arm
def _cpu_worker(args):
    """One host core: step one oracle env (restated reference path) with U(-1,1) actions for `n_steps` steps."""
    wid, n_steps, warm = args
    import numpy as np
    from oracle import harness      # the cpu_baseline / reference arm is the one place bench.py may run the oracle
    env = harness.make_env("restated", harness.config_path(), CONFIG_KW, SIM_KW)
    run = harness.OracleRunner(env, seed=1234, env_id=wid)
    run.reset()
    rng = np.random.RandomState(wid)
    for _ in range(warm):
        run.step(rng.uniform(-1, 1, 3))
    t0 = time.perf_counter()
    for _ in range(n_steps):
        run.step(rng.uniform(-1, 1, 3))
    dt = time.perf_counter() - t0
    k = sum((n - 2) // 6 for n in run.nfev[warm:])
    return n_steps, dt, k


def cpu_reference_rate(seconds=None, cores=None, n_steps=None, warm=5):
    """Time the CPU oracle (kind "port": the restated reference path — /root/reference and PyFly do not exist on the
    GPU box) with one process per host core, the SubprocVecEnv topology of train_rl_controller.py:223 (without its
    per-step pipe synchronisation, which only favours the CPU number)."""
    import multiprocessing as mp
    cores = cores or os.cpu_count() or 1
    if n_steps is None:
        n_steps = max(20, int(seconds * 150.0))   # ~150 env-steps/s/core first guess sizes the bounded sample
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        t0 = time.perf_counter()
        res = pool.map(_cpu_worker, [(w, n_steps, warm) for w in range(cores)], chunksize=1)
        wall = time.perf_counter() - t0
    total = sum(r[0] for r in res)
    slowest = max(r[1] for r in res)
    return {"value": total / slowest, "unit": "env-steps/s", "cores": cores, "kind": "port",
            "sample": "%d procs x %d env steps of the bench workload, restated FixedWingAircraft+PyFly oracle "
                      "(scipy solve_ivp RK45), U(-1,1) actions; %.1f s wall; mean dopri5 attempts/step %.2f"
                      % (cores, n_steps, wall, sum(r[2] for r in res) / max(1, total))}, slowest


CPU_STEPS_PER_UNIT = 16   # reference arm: one bench "step" = every host core advances its env 16 env steps


def run_reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    base, slowest = cpu_reference_rate(cores=cores, n_steps=a.steps * CPU_STEPS_PER_UNIT,
                                       warm=max(3, a.warmup) * CPU_STEPS_PER_UNIT)
    line = {"impl": "reference", "metric": "env-steps/s", "value": base["value"], "unit": "env-steps/s",
            "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": 1e3 * slowest / a.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD + " — bounded CPU sample: one env per host core, %d env steps per bench step"
                       % CPU_STEPS_PER_UNIT},
            "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# -------------------------------------------------------------------------------------------------------- GPU arm
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.lines, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 8:
                continue
            try:
                sm.append(float(p[1]))
                mx.append(float(p[2]))
            except ValueError:
                continue
            for nme, val in zip(names, p[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(nme)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def run_gpu_arm(a):
    import numpy as np
    import torch
    import torch.distributed as dist
    import __graft_entry__ as ge

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly ONE line (the JSON): libraries that print to fd 1 (NCCL's version banner) go to stderr
    sys.stdout.flush()
    json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if world != a.gpus and world > 1:
        a.gpus = world
    torch.cuda.set_device(local)
    placement = None
    if world > 1 and os.environ.get("FWGYM_BENCH_BIND", "0") == "1":
        # Opt-in: one block of host cores per rank on the NUMA node of its GPU, chosen before any pinned host memory
        # exists.  OFF by default: this pool's 8-GPU boxes are VMs with one virtual NUMA node and no GPU affinity in sysfs,
        # where pinning ranks to core blocks LOWERED the concurrent device -> host bandwidth (12.9 / 21 GB/s per GPU
        # against 18 / 42 GB/s unpinned; scripts/gpu_d2h_concurrent.py, profiles/r2_n8_d2h_concurrent.txt)
        from fwgym_b200.parallel import bind_to_gpu_numa_node
        placement = bind_to_gpu_numa_node(local, world)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if rank == 0:
        ge.build()
    if world > 1:
        dist.barrier()
    from fwgym_b200 import FixedWingVecEnv, _capi
    from fwgym_b200.config import DEFAULT_ENV_CONFIG

    n = a.envs_per_gpu
    vec = FixedWingVecEnv(DEFAULT_ENV_CONFIG, n, device=dev, config_kw=CONFIG_KW, sim_config_kw=SIM_KW,
                          seed=20261017, env_offset=rank * n)
    vec.reset()
    gen = torch.Generator(device=dev)
    gen.manual_seed(1 + rank)
    prof_steps_n = min(a.steps, 20)
    total = a.warmup + a.steps + prof_steps_n
    # synthetic policy output: i.i.d. U(-1,1) actions, a fresh batch per step, resident in HBM before timing
    actions = torch.rand((total, n, 3), generator=gen, device=dev, dtype=torch.float32) * 2 - 1
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2
    burn_actions = torch.rand((16, n, 3), generator=gen, device=dev, dtype=torch.float32) * 2 - 1

    def burn_in():
        for i in range(a.burn_in):
            vec.step_tensors(burn_actions[i % 16])
        torch.cuda.synchronize(dev)
    flush_mode = os.environ.get("FWGYM_BENCH_FLUSH", "write")
    flush_rd = torch.zeros(64 * 1024 * 1024, dtype=torch.int32, device=dev) if flush_mode == "write+read" else None

    def flush_l2():
        # write a buffer larger than L2.  "write+read" (diagnostic): a 256 MiB read pass behind it, so that the lines the
        # memset leaves DIRTY in L2 are written back before the timed step starts instead of on its misses
        flush.zero_()
        if flush_rd is not None:
            flush_rd.sum()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    burn_in()
    for i in range(a.warmup):
        vec.step_tensors(actions[i])
    vec.reset_counters()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
    barrier()
    t_wall0 = time.perf_counter()
    for k in range(a.steps):
        flush_l2()                          # L2 flush between timed iterations (not inside the timed interval)
        ev[k][0].record()
        last = vec.step_tensors(actions[a.warmup + k])
        ev[k][1].record()
    barrier()
    wall = time.perf_counter() - t_wall0
    if a.dump_outputs and rank == 0:        # the env's output buffers: the passes below overwrite them
        obs, rew, done, term = (x.cpu().numpy() for x in last)
        dump_outputs(a.dump_outputs, {"obs": obs, "reward": rew, "done": done.astype(np.float32),
                                      "term": term.astype(np.float64)})
    step_ms = sorted(e0.elapsed_time(e1) for e0, e1 in ev)
    ms = sum(step_ms)
    ctr = vec.counters()
    clocks = sampler.stop() if rank == 0 else None
    # per-kernel times for the roofline: a separate pass with an event between the dynamics kernels and the env
    # kernel (that event serialises the two; in the timed region above the env kernel runs as a programmatic dependent
    # of the attempt kernel and overlaps its tail)
    vec.set_profiling(True)
    k_hist = torch.zeros(64, dtype=torch.int64, device=dev)     # dopri5 attempts per env step; bin 63 = 63 and more
    k_max = torch.zeros((), dtype=torch.int32, device=dev)
    for k in range(prof_steps_n):
        flush_l2()
        vec.step_tensors(actions[a.warmup + a.steps + k])
        la = vec.last_attempts()
        k_hist += torch.bincount(la.clamp(max=63).long(), minlength=64)
        k_max = torch.maximum(k_max, la.max())
    dyn_ms, env_ms, prof_steps = vec.profile()
    vec.set_profiling(False)
    ctr_prof = vec.counters()
    msum_local = vec.metric_sums()        # episode metric sums of the device-resident passes
    launches_per_step = vec.launches_per_step
    prof_env_steps = ctr_prof["env_steps"] - ctr["env_steps"]
    prof_attempts = ctr_prof["attempts"] - ctr["attempts"]

    # ---- opt-in fp32 dynamics, stated separately (not part of the fp64 parity claim): same workload, same timing rules
    vec32 = FixedWingVecEnv(DEFAULT_ENV_CONFIG, n, device=dev, config_kw=CONFIG_KW, sim_config_kw=SIM_KW,
                            seed=20261017, env_offset=rank * n, precision="fp32")
    vec32.reset()
    for i in range(a.burn_in):
        vec32.step_tensors(burn_actions[i % 16])
    for i in range(a.warmup):
        vec32.step_tensors(actions[i])
    ev32 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
    barrier()
    for k in range(a.steps):
        flush_l2()
        ev32[k][0].record()
        vec32.step_tensors(actions[a.warmup + k])
        ev32[k][1].record()
    barrier()
    ms32 = sum(e0.elapsed_time(e1) for e0, e1 in ev32)
    vec32.close()

    # ---- second workload, stated separately (VERDICT r1: the headline workload flies random actions into constraint
    # failures, so steps_max / success paths never run in its timed region): the reference's EVALUATION setting at scale -
    # examples/fixed_wing_config.json with evaluate_controller.py:68-79's overrides (episode ends on a 100-step success
    # streak, steps_max 1500, physical actions) flown by the reference's PID controller (evaluate_controller.py:141-151;
    # fw_pid_step on the device), same turbulence, same envs per GPU, same L2 flush / events.  The
    # burn-in is longer (>= 600 steps) so that episode ages are mixed: PID episodes last 200-300 steps.
    from fwgym_b200.evaluate import DevicePID, EVAL_CONFIG_KW
    ckw_pid = dict(EVAL_CONFIG_KW)                 # (that config has no observation-noise entry: none here)
    ckw_pid["action"] = {"scale_space": False}
    cfg_pid = os.path.join(os.path.dirname(DEFAULT_ENV_CONFIG), "fixed_wing_config_examples.json")
    vecp = FixedWingVecEnv(cfg_pid, n, device=dev, config_kw=ckw_pid, sim_config_kw=SIM_KW,
                           seed=20261017, env_offset=rank * n)
    pid = DevicePID(vecp)
    vecp.reset()
    pid_done = None
    pid_burn = max(a.burn_in, 600) if a.burn_in > 0 else 0
    for i in range(pid_burn + a.warmup):
        _, _, pid_done, _ = vecp.step_tensors(pid(pid_done))
    vecp.reset_counters()
    msum_p0 = vecp.metric_sums()
    evp = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
    kp_max = torch.zeros((), dtype=torch.int32, device=dev)
    barrier()
    for k in range(a.steps):
        flush_l2()
        evp[k][0].record()
        _, _, pid_done, _ = vecp.step_tensors(pid(pid_done))   # controller launch + env step inside the timed interval
        evp[k][1].record()
        kp_max = torch.maximum(kp_max, vecp.last_attempts().max())
    barrier()
    msp = sum(e0.elapsed_time(e1) for e0, e1 in evp)
    ctr_p = vecp.counters()
    msum_p = vecp.metric_sums() - msum_p0
    pid_variant = vecp.kernel_variant()
    vecp.close()

    # ---- end-to-end through the public API with HOST buffers (fwgym_b200.HostStepper over the C-ABI fw_host_submit /
    # fw_host_wait): every step moves its actions pinned-host -> device and its observations / rewards / dones /
    # termination codes device -> pinned-host.  Three call patterns, all from a fresh reset + the same burn-in:
    #   closed loop, two half-batches ping-ponged (THE e2e value): a policy needs obs_t before it can send a_{t+1}
    #     (evaluate_controller.py:153-154, train_rl_controller.py:223), so each half-batch handle has ONE step in flight
    #     and its next submit happens only after its previous results are on the host; while half A's results travel and
    #     the host turns them around, half B's kernels run.
    #   closed loop, one handle, depth 1: the same dependency without the second half: the GPU idles during the copies.
    #   open loop, depth 2 (round 1's number): action t+1 is sent before observation t is read - an upper bound no
    #     policy can use.
    from fwgym_b200 import HostStepper
    e2e_steps = a.e2e_steps or a.steps
    n_act = 48
    host_actions = (torch.rand((n_act, n, 3)) * 2 - 1).pin_memory()
    checksum = 0.0
    host_split = [0.0, 0.0]     # seconds inside submit() / wait() of the ping-pong pass (diagnostics)

    def e2e_open(stepper, first, count):
        nonlocal checksum
        pending = []
        for i in range(count):
            pending.append(stepper.submit(host_actions[(first + i) % n_act]))
            if len(pending) == stepper.depth:
                obs, rew, done = stepper.wait(pending.pop(0))
                checksum += float(rew[0])          # touch the host result of every step
        while pending:
            obs, rew, done = stepper.wait(pending.pop(0))
            checksum += float(rew[0])

    def timed(fn, warm, count):
        fn(0, warm)
        barrier()
        t0 = time.perf_counter()
        fn(warm, count)
        torch.cuda.synchronize(dev)
        local = time.perf_counter() - t0       # this rank's own time (the reported one is the max over ranks)
        barrier()
        return time.perf_counter() - t0, local

    # (c) open loop, depth 2, and (b) closed loop depth 1 on the full-batch handle
    # closed loops: results written by the env kernel straight into mapped pinned host memory (no D2H copy behind the
    # step; +12 % measured); the open loop keeps the copy, which overlaps the NEXT step's kernels there
    zc = os.environ.get("FWGYM_HOST_ZEROCOPY", "1") == "1"
    stepper2 = HostStepper(vec, depth=int(os.environ.get("FWGYM_HOST_DEPTH", "2")), zero_copy=False)
    vec.reset()
    burn_in()
    open_s, _ = timed(lambda f, c: e2e_open(stepper2, f, c), a.warmup, e2e_steps)
    stepper2.close()
    stepper1 = HostStepper(vec, depth=1, zero_copy=zc)
    vec.reset()
    burn_in()
    d1_s, _ = timed(lambda f, c: e2e_open(stepper1, f, c), a.warmup, e2e_steps)
    stepper1.close()
    h2d_bytes, d2h_bytes = stepper1.h2d_bytes, stepper1.d2h_bytes
    vec.close()

    # (a) two half-batch handles (global env ids [rank*n, rank*n + n/2) and [rank*n + n/2, (rank+1)*n)), one stream each
    parts = int(os.environ.get("FWGYM_E2E_PARTS", "2"))      # sub-batch handles per rank (2 measured best, DESIGN.md §6)
    bounds = [n * j // parts for j in range(parts + 1)]
    halves, steppers, streams = [], [], []
    for j in range(parts):
        v = FixedWingVecEnv(DEFAULT_ENV_CONFIG, bounds[j + 1] - bounds[j], device=dev, config_kw=CONFIG_KW,
                            sim_config_kw=SIM_KW, seed=20261017, env_offset=rank * n + bounds[j])
        st = torch.cuda.Stream(device=dev)
        with torch.cuda.stream(st):
            v.reset()
            for i in range(a.burn_in):
                v.step_tensors(burn_actions[i % 16][bounds[j]:bounds[j + 1]])
        halves.append(v); streams.append(st); steppers.append(HostStepper(v, depth=1, zero_copy=zc))
    torch.cuda.synchronize(dev)
    half_actions = [host_actions[:, bounds[j]:bounds[j + 1]] for j in range(parts)]
    half_actions = [torch.empty_like(h).copy_(h).pin_memory() for h in half_actions]   # contiguous per part

    def e2e_pingpong(first, count):
        nonlocal checksum
        slots = [None] * parts
        for i in range(count + 1):
            for j in range(parts):
                tb = time.perf_counter()
                if slots[j] is not None:
                    obs, rew, done = steppers[j].wait(slots[j])      # obs_t of this half is on the host ...
                    checksum += float(rew[0]) + float(obs[0, 0])
                    slots[j] = None
                tc = time.perf_counter()
                host_split[1] += tc - tb
                if i < count:
                    with torch.cuda.stream(streams[j]):               # ... before its a_{t+1} is sent
                        slots[j] = steppers[j].submit(half_actions[j][(first + i) % n_act])
                    host_split[0] += time.perf_counter() - tc

    e2e_pingpong(0, a.warmup)
    barrier()
    host_split[0] = host_split[1] = 0.0
    t0 = time.perf_counter()
    e2e_pingpong(a.warmup, e2e_steps)
    torch.cuda.synchronize(dev)
    e2e_local = time.perf_counter() - t0
    barrier()
    e2e_s = time.perf_counter() - t0
    half_watchdog = sum(v.counters()["watchdog"] for v in halves)

    place_all = [placement]
    if world > 1:
        place_all = [None] * world
        dist.all_gather_object(place_all, placement)
    tt = torch.tensor([ms, e2e_s * 1e3, dyn_ms, env_ms, wall * 1e3, open_s * 1e3, d1_s * 1e3, step_ms[-1], ms32, msp],
                      dtype=torch.float64, device=dev)
    cnt = torch.tensor([ctr["env_steps"], ctr["attempts"], ctr["warp_max_attempts"], ctr["warp_steps"],
                        ctr["failures"], ctr["resets"], prof_env_steps, prof_attempts,
                        ctr_prof["watchdog"] + half_watchdog],
                       dtype=torch.float64, device=dev)
    msum = torch.tensor(msum_local, dtype=torch.float64, device=dev)
    pidc = torch.tensor([ctr_p["env_steps"], ctr_p["attempts"]] + [float(x) for x in msum_p], dtype=torch.float64, device=dev)
    kp_max_t = kp_max.to(torch.float64).reshape(1)
    e2e_each = [e2e_local * 1e6 / e2e_steps]
    if world > 1:
        g = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(g, torch.tensor([e2e_each[0]], dtype=torch.float64, device=dev))
        e2e_each = [float(x.item()) for x in g]
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)     # time = max over ranks
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
        dist.all_reduce(msum, op=dist.ReduceOp.SUM)   # the only data-path collective: episode metric sums
        dist.all_reduce(pidc, op=dist.ReduceOp.SUM)
        dist.all_reduce(kp_max_t, op=dist.ReduceOp.MAX)
    ms, e2e_ms, dyn_ms, env_ms, wall_ms, open_ms, d1_ms, step_max_ms, ms32, msp = tt.tolist()
    env_steps, attempts, wmax, wsteps, failures, resets, p_env_steps, p_attempts, watchdog = cnt.tolist()
    if rank == 0:
        total_env_steps = float(n) * a.steps * world
        e2e_env_steps = float(n) * e2e_steps * world
        value = total_env_steps / (ms * 1e-3)
        pct = lambda q: step_ms[min(len(step_ms) - 1, int(q * len(step_ms)))]
        kh = k_hist.cpu().numpy()
        k_mean = attempts / max(1.0, env_steps)
        # roofline of the dominant kernel (dynamics, FP64 pipe): algorithmic flops of ONE rank / its kernel time
        fl = ctypes.c_double()
        pk_ms = ctypes.c_double()
        _capi.check(_capi.lib().fw_dfma_peak(local, ctypes.byref(fl), ctypes.byref(pk_ms)))
        flops_rank = (F_FIXED * p_env_steps + F_ATTEMPT * p_attempts) / world   # of the profiled pass
        achieved = flops_rank / (dyn_ms * 1e-3) / 1e12
        # DRAM traffic cannot be measured outside a profiler: the number is COPIED from the committed ncu capture named
        # in traffic_from (profiles/traffic.json says which file, commit and workload), it is not a live measurement
        traffic, ncu_notes, traffic_from = None, None, None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.isfile(tpath):
            with open(tpath) as f:
                tj = json.load(f)
            traffic, ncu_notes = tj.get("dyn_kernel_dram_bytes_per_launch"), tj.get("ncu")
            traffic_from = tj.get("from")
        line = {
            "metric": "env-steps/s", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "envs_per_gpu": n, "actions": "i.i.d. U(-1,1)^3 per step", "burn_in_steps": a.burn_in,
                       "l2": "256 MiB memset between timed steps; per-step CUDA events summed"
                             + ("; + 256 MiB read pass (memset's dirty lines written back before the step)"
                                if flush_mode == "write+read" else ""),
                       "parallelism": "env-sharded x%d, no step-path collective" % world},
            "clocks": clocks,
            "step_ms": {"p50": pct(0.5), "p99": pct(0.99), "max_rank0": step_ms[-1], "max_any_rank": step_max_ms,
                        "min": step_ms[0], "note": "per-step CUDA-event times of the timed region on rank 0: rare dopri5 "
                        "stragglers (attempts_per_env_step.max) stretch single steps"},
            "e2e": {"value": e2e_env_steps / (e2e_ms * 1e-3), "unit": "env-steps/s",
                    "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes, "steps": e2e_steps,
                    "pattern": "closed loop: 2 half-batch handles per GPU ping-ponged, one step in flight each; a "
                               "half's a_{t+1} is submitted only after its obs_t / reward_t / done_t are in host memory",
                    "zero_copy_results": zc,
                    "closed_loop_depth1": {"value": e2e_env_steps / (d1_ms * 1e-3),
                                           "pattern": "one handle, one step in flight (GPU idle during copies)"},
                    "open_loop_depth2": {"value": e2e_env_steps / (open_ms * 1e-3),
                                         "pattern": "round 1's figure: a_{t+1} sent before obs_t is read; an upper bound "
                                                    "no policy can use"},
                    "us_per_step_by_rank": [round(x, 1) for x in e2e_each],
                    "host_placement_by_rank": place_all,
                    "rank0_host_us_per_step": {"submit": round(host_split[0] * 1e6 / e2e_steps, 1),
                                               "wait": round(host_split[1] * 1e6 / e2e_steps, 1)},
                    "how": "C-ABI fw_host_open_ex / fw_host_submit / fw_host_wait (HostStepper): actions copied from pinned "
                           "host memory every step; observations / rewards / dones / termination codes land in pinned host "
                           "memory every step - closed loops: written there by the env kernel itself (mapped memory, "
                           "coalesced through a shared-memory tile), open loop: one device -> host copy on its own stream; "
                           "wall clock over %d steps after %d warm-up steps" % (e2e_steps, a.warmup)},
            "fp32_mode": {"value": total_env_steps / (ms32 * 1e-3), "unit": "env-steps/s", "dtype": "f32",
                          "ms_per_step": ms32 / a.steps,
                          "note": "precision='fp32' dynamics kernels on the same workload, same steps / flush / events; "
                                  "stated separately: fp32 adaptive stepping is not held to the 1e-9 parity bar (integer "
                                  "state still is, tests/test_gpu_parity.py::test_fp32_mode_feature_config_integer_state)"},
            "controlled_flight": {
                "value": total_env_steps / (msp * 1e-3), "unit": "env-steps/s", "dtype": "f64", "ms_per_step": msp / a.steps,
                "workload": "the reference's evaluation setting at scale: examples/fixed_wing_config.json + "
                            "evaluate_controller.py:68-79 overrides (success streak 100 -> done, steps_max 1500, physical "
                            "actions), PID controller on the device (fw_pid_step, one launch per step inside the timed "
                            "interval), turbulence moderate, %d envs/GPU, %d burn-in steps" % (n, pid_burn),
                "kernels": pid_variant,
                "mean_attempts_per_env_step": pidc[1].item() / max(1.0, pidc[0].item()),
                "max_attempts_per_env_step": int(kp_max_t.item()),
                "episodes_in_timed_region": {"finished": pidc[2].item(), "successes": pidc[3].item(),
                                             "failures": pidc[6].item(), "ended_on_steps_max": pidc[7].item(),
                                             "ended_on_success": pidc[8].item(),
                                             "mean_length": pidc[5].item() / max(1.0, pidc[2].item())},
                "note": "stated separately from `value` (BASELINE configs[2] is the random-action workload): here the "
                        "aircraft are flown to their targets, so the success / steps_max terminations and their resets run "
                        "inside the timed region"},
            "gpu_launches": int(launches_per_step * a.steps),
            "roofline": {"bound": "fp64", "achieved": achieved, "peak": fl.value / 1e12, "unit": "TFLOP/s",
                         "frac": achieved / (fl.value / 1e12), "traffic": traffic, "traffic_from": traffic_from,
                         "peak_source": "DFMA micro-benchmark run in this process (fw_dfma_peak); MEASURED_PEAKS.json "
                                        "has no FP64 entry",
                         "kernel": "fw_init_kernel + fw_attempt_kernel <double> (the simulator step; timed together)",
                         "kernel_ms_per_launch": dyn_ms / max(1, prof_steps),
                         "kernel_share_of_step": dyn_ms / max(1e-9, dyn_ms + env_ms),
                         "how": "%d extra steps with an event between the dynamics and env kernels (serialised); the "
                                "timed region runs them overlapped" % prof_steps,
                         "flops_per_env_step": "1080 + 3660*k, k = dopri5 attempts counted on device",
                         "ncu_capture": ncu_notes,   # ditto: from the committed capture, not live
                         "mean_attempts_per_env_step": k_mean,
                         "attempts_per_env_step": {"histogram_1_to_16": [int(x) for x in kh[1:17]],
                                                   "more_than_16": int(kh[17:].sum()), "zero": int(kh[0]),
                                                   "max": int(k_max.item()), "over": "%d profiled steps" % prof_steps},
                         "warp_divergence": {"warp_passes": wmax / world, "lane_attempts": wsteps / world,
                                             "lane_efficiency": wsteps / max(1.0, 32.0 * wmax)}},
            "env_kernel": {"bound": "hbm", "ms_per_launch": env_ms / max(1, prof_steps),
                           "achieved_gbs": ENV_BYTES_PER_STEP * n / max(1e-9, env_ms / max(1, prof_steps) * 1e-3) / 1e9,
                           "peak_gbs": _measured_peaks().get("hbm_gbs"),
                           "note": "time between two CUDA events around the launch of the serialised profiling pass; "
                                   "in the timed region the kernel runs overlapped with the attempt kernel's tail and its "
                                   "last block ends ~25 us behind the attempt kernel on the GPU's own timer "
                                   "(profiles/r2f_step_timeline.txt); latency-bound, not bandwidth-bound"},
            "wall_ms_timed_region": wall_ms,
            "overlap": {"env_kernel": "programmatic dependent launch behind the attempt kernel, per-chunk completion "
                                      "counters", "serial_ms_per_step": (dyn_ms + env_ms) / max(1, prof_steps),
                        "watchdog": watchdog},
            "episodes": {"finished": msum[0].item(), "failures": msum[4].item(), "resets": resets},
        }
        if world == 1 and not a.no_cpu_baseline:
            line["cpu_baseline"] = cpu_reference_rate(a.cpu_baseline_seconds)[0]
        json_out.write(json.dumps(line) + "\n")
        json_out.flush()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def _measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        with open(p) as f:
            return json.load(f)
    return {"hbm_gbs": 6650.0, "source": "fallback"}


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)
