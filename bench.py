#!/usr/bin/env python
"""bench.py — env-steps/s of batched CubicEnv.step on B200 (BASELINE.json metric), one JSON line on stdout.

    python bench.py [--gpus N --steps K --warmup W] [--workload c4|c2|c3] [--impl reference] [--dump-outputs DIR]

A "step" is ONE nav3d_step launch over every env of the workload (one pass of the hot path over one batch):
  value     device-resident: actions already in HBM, observations written into an HBM rollout ring; CUDA-event timed
  e2e       the same step through nav3d_step_host with pinned HOST buffers (actions H2D, obs/reward/flags D2H, every step)
  roofline  algorithmic bytes (592 B per env-step, SURVEY §8d / DESIGN.md §5) x envs per launch / mean launch duration
  cpu_baseline  the Python port of the reference env (oracle/py_cubic.py) on this box's host cores, plus the C oracle
Workloads (BASELINE.json configs): c4 = 2^20 envs sharded over the N GPUs (default, the config the 1/2/4/8 metric is
quoted on), c2 = 4096 envs on P1_training, c3 = 65536 envs on P2+P3_training.  Under torchrun every rank holds its own
env shard and room table; there is no collective on the data path.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
import _nav3d_path  # noqa: E402,F401

B_ALG = {10: 592, 4: 516}          # algorithmic bytes per env-step, SURVEY.md §8d
METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"


def workload_spec(name):
    if name == "c4":
        return dict(name="c4", envs_total=1 << 20, room_dirs=["P1_training"], L=10, scaling="strong",
                    desc="BASELINE configs[3]: 2^20 CubicEnv envs env-sharded over the GPUs, rooms/P1_training (5 rooms), "
                         "L=10, uniform random actions, auto-reset")
    if name == "c2":
        return dict(name="c2", envs_total=4096, room_dirs=["P1_training"], L=10, scaling="weak",
                    desc="BASELINE configs[1]: 4096 CubicEnv envs per GPU, rooms/P1_training, L=10, random actions")
    if name == "c3":
        return dict(name="c3", envs_total=65536, room_dirs=["P2_training", "P3_training"], L=10, scaling="weak",
                    desc="BASELINE configs[2]: 65536 CubicEnv envs per GPU, rooms/P2_training + P3_training (42 rooms), L=10")
    if name == "s4":
        return dict(name="s4", envs_total=1 << 20, room_dirs=["P1_training"], L=4, scaling="strong", simple=True,
                    desc="2^20 simpleEnv envs (envs/simpleEnv.py) env-sharded over the GPUs, rooms/P1_training, L=4, "
                         "uniform random actions, auto-reset")
    raise SystemExit(f"unknown workload {name}")


def load_rooms(spec):
    from nav3d.rooms import load_room_dir
    rooms = []
    for d in spec["room_dirs"]:
        rooms += load_room_dir(ROOT / "rooms" / d, sort=True, simple=bool(spec.get("simple")))
    return rooms


# ---------------------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE,
                                      stderr=subprocess.DEVNULL, text=True)
        except Exception:  # noqa: BLE001
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:  # noqa: BLE001
            self.p.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------
# CPU arms
# ---------------------------------------------------------------------------------------------------------------
def python_port_rate(grids, L, steps_per_worker, workers):
    """N worker processes, one env each (the reference's SubprocVecEnv shape); returns (steps/s summed, wall seconds)."""
    import multiprocessing as mp
    from oracle.py_cubic import worker_rollout
    ctx = mp.get_context("fork")
    t0 = time.perf_counter()
    with ctx.Pool(workers) as pool:
        res = pool.map(worker_rollout, [(grids, L, steps_per_worker, 42 + i) for i in range(workers)])
    wall = time.perf_counter() - t0
    return sum(n / t for n, t in res), wall


def c_port_rate(rooms, L, n_envs, T, threads):
    from oracle import c_oracle
    orooms = [c_oracle.OracleRoom(r.grid, -2) for r in rooms]
    ov = c_oracle.OracleVec(n_envs, orooms, L, -2.0, 0, 0, True)
    c_oracle.set_threads(threads)
    ov.reset()
    ov.rollout_random(8, 0)
    t0 = time.perf_counter()
    n, _, _ = ov.rollout_random(T, 8)
    dt = time.perf_counter() - t0
    c_oracle.set_threads(1)
    return n / dt


def load_rooms_standalone(spec):
    """The room grids WITHOUT importing the product package: nav3d/__init__.py dlopens libnav3d_b200.so, which the
    reference arm must not map.  rooms.py itself only needs NumPy, so it is loaded as a lone module."""
    import importlib.util
    mspec = importlib.util.spec_from_file_location("nav3d_rooms_standalone", _nav3d_path.PKG_DIR / "nav3d" / "rooms.py")
    mod = importlib.util.module_from_spec(mspec)
    sys.modules[mspec.name] = mod
    mspec.loader.exec_module(mod)
    rooms = []
    for d in spec["room_dirs"]:
        rooms += mod.load_room_dir(ROOT / "rooms" / d, sort=True, simple=bool(spec.get("simple")))
    return rooms


def cpu_arm(spec, steps_per_worker, workers, one_process_steps=0):
    """The CPU implementation of the path on this box's host cores, one env per worker process (the reference's own
    SubprocVecEnv shape, train/Grid_Train.py:191-192).  kind "reference": the UNMODIFIED reference class from oracle/_ref
    (staged by __graft_entry__.build() where /root/reference exists), resets and their file parse included (BASELINE.md §3);
    kind "port": oracle/py_cubic.py, only when oracle/_ref is absent.  Returns (rate, wall, one_process_rate, kind, what)."""
    from oracle import ref_runner
    if ref_runner.available() and not spec.get("simple") and len(spec["room_dirs"]) == 1:
        room_dir = ROOT / "rooms" / spec["room_dirs"][0]
        rate, wall = ref_runner.reference_rate(room_dir, spec["L"], steps_per_worker, workers)
        one = ref_runner.reference_rate(room_dir, spec["L"], one_process_steps, 1)[0] if one_process_steps else None
        return rate, wall, one, "reference", ("the unmodified reference envs/CubicEnv.py GridAgent (oracle/_ref, behind the "
                                               "gymnasium/matplotlib import shims of SURVEY Appendix A), reset(seed=42+rank) "
                                               "then reset() on every episode end inside the timed region, stdout redirected")
    grids = [r.grid.astype(int) for r in load_rooms_standalone(spec)]
    rate, wall = python_port_rate(grids, spec["L"], steps_per_worker, workers)
    one = python_port_rate(grids, spec["L"], one_process_steps, 1)[0] if one_process_steps else None
    return rate, wall, one, "port", "oracle/py_cubic.py (Python port; oracle/_ref absent, so the reference itself could not be timed)"


def run_reference(args):
    """The reference arm: the reference's own CPU implementation of the path on all host cores — the unmodified
    envs/CubicEnv.py class (oracle/_ref), one env per worker process like the reference's SubprocVecEnv.  Nothing of the
    product (nav3d package, libnav3d_b200.so) is imported here."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    spec = workload_spec(args.workload)
    cores = os.cpu_count() or 1
    K, W = args.steps, args.warmup
    # each "step" = every worker advances its env by S env-steps; S sized so the whole run takes about a minute
    S = int(max(20, min(4000, 60.0 * 5000.0 / max(1, K + W))))
    cpu_arm(spec, max(1, W * S // 4), cores)                               # warm-up (fork, page-in)
    rate, wall, one, kind, what = cpu_arm(spec, K * S, cores, one_process_steps=min(K * S, 10000))
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": K, "warmup": W,
        "ms_per_step": 1e3 * wall / K, "higher_is_better": True, "scaling": spec["scaling"], "vs_baseline": None,
        "dtype": "python int/f64 (NumPy)", "data": "synthetic",
        "config": {"workload": spec["desc"],
                   "sample": f"{cores} worker processes x 1 env, {S} env-steps per worker per step: a bounded CPU sample of the "
                             f"{spec['envs_total']}-env workload (same rooms, L and action distribution; NOT the same env count)",
                   "same_config": False},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": f"{what}; {cores} processes x {K * S} random-action steps", "one_process": one},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------
class StepBuffers:
    """Device-resident operands of the timed loop: a ring of action rows, a ring of observation buffers, reward and flags."""
    def __init__(self, eng, n, torch, ring=4, act_rows=16, seed=0):
        # act_rows: one row of uniform random actions per step where memory allows (<= 1024 rows = 8 GB at 2^20 envs).  A short
        # ring makes every env repeat a 16-step pattern: it drifts into a wall and keeps bumping there, and the "random-action"
        # step becomes cheaper with every period (tools/per_launch.py).
        dev = eng.device
        g = torch.Generator(device=dev).manual_seed(1234 + seed)
        self.ring, self.act_rows = ring, act_rows
        self.actions = torch.randint(0, 6, (act_rows, n), generator=g, device=dev, dtype=torch.int64)
        self.obs = torch.empty((ring, n, eng.obs_dim), dtype=torch.float32, device=dev)
        self.rew = torch.empty(n, dtype=torch.float32, device=dev)
        self.te = torch.empty(n, dtype=torch.uint8, device=dev)
        self.tr = torch.empty(n, dtype=torch.uint8, device=dev)
        self.t = 0                                  # steps taken since the reset

    def step(self, eng):
        eng.step(self.actions[self.t % self.act_rows], self.obs[self.t % self.ring], self.rew, self.te, self.tr)
        self.t += 1

    def last_obs(self):
        return self.obs[(self.t - 1) % self.ring]


def timed_steps(eng, buf, steps, torch, dist, world):
    """CUDA-event timing of `steps` nav3d_step launches on the engine's stream, barrier + synchronize on both sides, max over
    ranks.  Returns (ms_total_max_over_ranks, ms_total_local, launches)."""
    dev = eng.device
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    l0 = eng.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(steps):
        buf.step(eng)
    e1.record()
    torch.cuda.synchronize(dev)
    ms_local = e0.elapsed_time(e1)
    ms = ms_local
    if world > 1:
        dist.barrier()
        tmax = torch.tensor([ms_local], device=dev, dtype=torch.float64)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ms = float(tmax.item())
    return ms, ms_local, eng.launch_count - l0


DUMP_MAX_ENVS = 1 << 17            # 2^17 envs x (80 + 3) f32 + f64 id = 44.6 MB, under the 64 MB a dump may take


def dump_outputs(out_dir, buf, torch):
    """Writes what the last timed nav3d_step returned to its caller (observation, reward, terminated, truncated) as
    float32 .npy files, for the envs of a fixed sample (seeded, the same in every run: all envs when at most
    DUMP_MAX_ENVS), plus their env ids (float64).  Two builds run with the same arguments can be compared file for
    file."""
    import numpy as np
    n = buf.rew.shape[0]
    if n <= DUMP_MAX_ENVS:
        idx = np.arange(n)
    else:
        idx = np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_ENVS, replace=False))
    tid = torch.as_tensor(idx, device=buf.rew.device)
    arrays = {"obs": buf.last_obs()[tid], "reward": buf.rew[tid], "terminated": buf.te[tid], "truncated": buf.tr[tid]}
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, t in arrays.items():
        np.save(out_dir / f"{name}.npy", t.cpu().numpy().astype(np.float32))
    np.save(out_dir / "env_ids.npy", idx.astype(np.float64))


def time_steps(eng, n, steps, warmup, torch, dist, world, lanes_note=None, ring=4, act_rows=16, seed=0):
    """Reset, `warmup` untimed steps, `steps` timed ones.  Returns (ms_total_max_over_ranks, ms_total_local, launches)."""
    buf = StepBuffers(eng, n, torch, ring, act_rows, seed)
    eng.reset(buf.obs[0])
    for _ in range(warmup):
        buf.step(eng)
    return timed_steps(eng, buf, steps, torch, dist, world)


class OracleSample:
    """A strided sample of the job's envs replayed by the C oracle (the parity checker, oracle/nav3d_oracle.c) under the
    same global env ids, Philox streams and actions: ties the timed number to correct output (VERDICT r1 item 2-iii)."""
    def __init__(self, rooms, L, seed, env_id0, n_local, k=256):
        import numpy as np
        from oracle import c_oracle
        self.np, self.c = np, c_oracle
        self.local = np.arange(3, n_local, max(1, n_local // k), dtype=np.int64)[:k]
        self.ov = c_oracle.OracleVec(len(self.local), [c_oracle.OracleRoom(r.grid, -2) for r in rooms], L, -2.0, seed, 0, True)
        self.ov.set_ids((self.local + env_id0).astype(np.uint32))
        self.ov.reset()
        self.steps = 0

    def replay(self, actions_rows, t_from, t_to):
        for t in range(t_from, t_to):
            self.ov.step(actions_rows[t % actions_rows.shape[0]][self.local])
        self.steps += t_to - t_from

    def replay_random(self, T, t0):
        self.ov.rollout_random_obs(T, t0)
        self.steps += T

    def compare(self, eng, obs, torch, what):
        np = self.np
        tid = torch.as_tensor(self.local, device=eng.device)
        got_obs = obs[tid].cpu().numpy()
        got_state = eng.get_state()[tid].cpu().numpy()[:, :15].astype(np.int64)
        ok_obs = bool(np.array_equal(got_obs.view(np.uint32), self.ov.obs.view(np.uint32)))
        ok_state = bool(np.array_equal(got_state, self.ov.state()))
        if not (ok_obs and ok_state):
            raise SystemExit(f"bench.py: {what}: the GPU result differs from the oracle replay (obs {ok_obs}, state {ok_state})")
        return {"envs_replayed": int(len(self.local)), "steps_replayed": int(self.steps), "obs_bit_exact": ok_obs,
                "state_equal": ok_state}


def time_steps_graph(eng, n, steps, torch, graph_len=50, ring=4, act_rows=16):
    """Same measurement with the step launches captured in a CUDA graph (graph_len steps per replay): what a trainer that
    graphs its rollout loop sees when the per-launch host overhead would otherwise dominate (small batches)."""
    dev = eng.device
    g = torch.Generator(device=dev).manual_seed(99)
    act_rows = max(act_rows, graph_len)
    actions = torch.randint(0, 6, (act_rows, n), generator=g, device=dev, dtype=torch.int64)
    obs = torch.empty((ring, n, 80), dtype=torch.float32, device=dev)
    rew = torch.empty(n, dtype=torch.float32, device=dev)
    te = torch.empty(n, dtype=torch.uint8, device=dev)
    tr = torch.empty(n, dtype=torch.uint8, device=dev)
    eng.reset(obs[0])
    for t in range(8):
        eng.step(actions[t % act_rows], obs[t % ring], rew, te, tr)
    torch.cuda.synchronize(dev)
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream(device=dev)
    with torch.cuda.graph(graph, stream=side):
        for t in range(graph_len):
            eng.step(actions[t % act_rows], obs[t % ring], rew, te, tr)
    reps = max(1, steps // graph_len)
    graph.replay()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        graph.replay()
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1), reps * graph_len


def affinity_from_smi(local_rank, bdf):
    """sysfs reports NUMA node -1 (virtualised PCI topology): fall back to the "CPU Affinity" column of `nvidia-smi topo -m`."""
    try:
        out = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=20).stdout.splitlines()
        clean = [__import__("re").sub(r"\x1b\[[0-9;]*m", "", ln) for ln in out]
        hdr = next(ln for ln in clean if "CPU Affinity" in ln)
        col = [c.strip() for c in hdr.split("\t")].index("CPU Affinity")
        row = next(ln for ln in clean if ln.startswith(f"GPU{local_rank}\t") or ln.startswith(f"GPU{local_rank} "))
        cell = [c.strip() for c in row.split("\t")][col]
        cpus = set()
        for part in cell.split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return f"gpu {bdf}: nvidia-smi topo affinity '{cell}' has no allowed cpu"
        if cpus == os.sched_getaffinity(0):
            return f"gpu {bdf}: sysfs NUMA -1; nvidia-smi topo affinity '{cell}' = all allowed cpus (single node: nothing to bind)"
        os.sched_setaffinity(0, cpus)
        return f"gpu {bdf}: sysfs NUMA -1; bound to nvidia-smi topo affinity '{cell}' ({len(cpus)} cpus)"
    except Exception as ex:  # noqa: BLE001
        return f"gpu {bdf}: no NUMA affinity reported by sysfs or nvidia-smi topo ({type(ex).__name__})"


def bind_to_gpu_numa_node(torch, local_rank):
    """Pin this process to the CPUs of the NUMA node the GPU hangs off, before any pinned host buffer is allocated
    (first-touch places the pages there): the end-to-end path is a PCIe copy of 342 MB per step per GPU, and a buffer on the
    other socket sends it across the inter-socket link as well.  Returns a short description for the JSON line."""
    try:
        p = torch.cuda.get_device_properties(local_rank)
        bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        node = int(Path(f"/sys/bus/pci/devices/{bdf}/numa_node").read_text().strip())
        if node < 0:
            return affinity_from_smi(local_rank, bdf)
        cpus = set()
        for part in Path(f"/sys/devices/system/node/node{node}/cpulist").read_text().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"gpu {bdf}: bound to NUMA node {node} ({len(cpus)} cpus)"
        return f"gpu {bdf}: NUMA node {node} has no allowed cpu"
    except Exception as ex:  # noqa: BLE001
        return f"not bound ({type(ex).__name__})"


def time_e2e(eng, n, steps, torch, dist, world):
    dev = eng.device
    a = [torch.randint(0, 6, (n,), dtype=torch.int64).pin_memory() for _ in range(4)]
    obs = torch.empty((n, eng.obs_dim), dtype=torch.float32).pin_memory()
    rew = torch.empty(n, dtype=torch.float32).pin_memory()
    te = torch.empty(n, dtype=torch.uint8).pin_memory()
    tr = torch.empty(n, dtype=torch.uint8).pin_memory()
    for t in range(3):
        eng.step_host(a[t % 4], obs, rew, te, tr)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for t in range(steps):
        eng.step_host(a[t % 4], obs, rew, te, tr)
    torch.cuda.synchronize(dev)
    sec = time.perf_counter() - t0
    if world > 1:
        dist.barrier()
        tmax = torch.tensor([sec], device=dev, dtype=torch.float64)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        sec = float(tmax.item())
    checksum = float(rew.sum())
    # the ceiling this path can reach on this host: plain pinned device->host copies of the same bytes, all ranks at once
    src = torch.empty((n, eng.obs_dim), dtype=torch.float32, device=dev)
    obs.copy_(src, non_blocking=True)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    reps = 5
    t0 = time.perf_counter()
    for _ in range(reps):
        obs.copy_(src, non_blocking=True)
    torch.cuda.synchronize(dev)
    csec = time.perf_counter() - t0
    if world > 1:
        dist.barrier()
        tmax = torch.tensor([csec], device=dev, dtype=torch.float64)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        csec = float(tmax.item())
    ceiling_gbs = world * reps * obs.numel() * 4 / csec / 1e9
    return sec, n * 8, n * (eng.obs_dim * 4 + 4 + 1 + 1), checksum, ceiling_gbs


def time_training(torch, dist, world, rank, local_rank, n_envs=16384, n_steps=128, iters=3):
    """BASELINE configs[4] (not roofline-graded): LSTM-PPO with the Grid_Train hyper-parameters on P1_training, env and
    rollout resident on the GPU, one rank per GPU with an NCCL gradient all-reduce per minibatch.  Weak scaling: every rank
    owns n_envs envs.  Returns env-steps/s over rollout + update, all ranks."""
    from nav3d import BatchedCubicEnv
    from nav3d.ppo import RecurrentPPO
    env = BatchedCubicEnv(ROOT / "rooms" / "P1_training", num_envs=n_envs, local_map_length=10, seed=42, sort_rooms=True,
                          device=local_rank, env_id0=rank * n_envs)
    model = RecurrentPPO(env, policy_kwargs=dict(net_arch=dict(pi=[256, 256, 128], vf=[256, 256, 128]), lstm_hidden_size=256,
                                                 n_lstm_layers=1),
                         learning_rate=3e-4, n_steps=n_steps, batch_size=(n_envs // 8) * n_steps, n_epochs=10, gamma=0.99,
                         gae_lambda=0.95, ent_coef=0.01, vf_coef=0.5, clip_range=0.2, seed=42)
    for _ in range(2):                  # warm-up: one eager rollout, then the CUDA-graph capture of the rollout
        model.collect_rollouts(); model.train()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t_roll = t_train = 0.0
    for _ in range(iters):
        t0 = time.perf_counter(); model.collect_rollouts(); torch.cuda.synchronize(); t1 = time.perf_counter()
        stats = model.train(); torch.cuda.synchronize(); t2 = time.perf_counter()
        t_roll += t1 - t0; t_train += t2 - t1
    sec = t_roll + t_train
    if world > 1:
        dist.barrier()
        tmax = torch.tensor([sec], device=env.device, dtype=torch.float64)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        sec = float(tmax.item())
    steps = iters * n_steps * n_envs * world
    out = {"workload": "BASELINE configs[4]: LSTM-PPO (MlpLstmPolicy 80->LSTM256 x2->256-256-128, Grid_Train hyper-parameters, "
                       f"{n_envs} envs x {n_steps} steps per GPU per rollout, 8 minibatches per epoch, 10 epochs) on P1_training, "
                       "GPU-resident env, NCCL gradient all-reduce per minibatch",
           "value": steps / sec, "unit": "env-steps/s (rollout + PPO update)", "iters": iters, "n_gpus": world,
           "rollout_share": t_roll / (t_roll + t_train), "rollout_steps_per_s_rank0": iters * n_steps * n_envs / t_roll,
           "minibatches_per_update": stats["minibatches"], "scaling": "weak"}
    env.close()
    del model
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", default="nav3d", choices=["nav3d", "reference"])
    ap.add_argument("--workload", default="c4", choices=["c4", "c2", "c3", "s4"])
    ap.add_argument("--lanes", type=int, default=0, help="lanes per env (0 = engine default)")
    ap.add_argument("--envs", type=int, default=0, help="override the total env count")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary workloads and the CPU baseline")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--preroll", type=int, default=600,
                    help="untimed fused random steps before the second, mid-episode measurement (0 = skip it)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what their last step returned (obs, reward, terminated, truncated "
                         "of a fixed sample of rank 0's envs, and the sample's env ids) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs saves what the GPU path's timed steps returned; the reference arm has none to save")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    from nav3d import Engine
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; nav3d has no CPU fallback")
    torch.cuda.set_device(local_rank)
    numa_note = bind_to_gpu_numa_node(torch, local_rank) if world > 1 else "single process: not bound"
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        import datetime
        # a rank that dies must not leave the others waiting for ten minutes in a collective
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(seconds=180))
    spec = workload_spec(args.workload)
    if args.envs:
        spec["envs_total"] = args.envs
    rooms = load_rooms(spec)
    L = spec["L"]
    if spec["scaling"] == "strong":
        n_total = spec["envs_total"]
        n_local = n_total // world
    else:
        n_local = spec["envs_total"]
        n_total = n_local * world
    eng = Engine(n_local, rooms, local_map_length=L, seed=2024, env_id0=rank * n_local, device=local_rank,
                 lanes_per_env=args.lanes, env_kind=1 if spec.get("simple") else 0)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    cubic = not spec.get("simple")
    # -- the regime the flags ask for: reset, W warm-up steps, K timed steps ("cold" when that is early in the episodes)
    n_rows = min(1024, args.warmup + 2 * args.steps)
    buf = StepBuffers(eng, n_local, torch, act_rows=n_rows)
    eng.reset(buf.obs[0])
    for _ in range(args.warmup):
        buf.step(eng)
    ms, ms_local, launches = timed_steps(eng, buf, args.steps, torch, dist, world)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, buf, torch)
    value = n_total * args.steps / (ms / 1e3)
    regime = "cold" if args.warmup + args.steps < 200 else "steady"
    check = None
    sample = None
    if cubic:
        sample = OracleSample(rooms, L, 2024, rank * n_local, n_local)
        sample.replay(buf.actions.cpu().numpy(), 0, buf.t)
        check = sample.compare(eng, buf.last_obs(), torch, "timed steps")
    # -- the same K steps mid-episode: a declared, untimed pre-roll of fused random steps, then K timed steps
    steady = None
    if cubic and args.preroll > 0:
        T = 40
        for i in range(args.preroll // T):
            eng.rollout_random(T, 1_000_000 + i * T, obs_last=buf.obs[0])
            sample.replay_random(T, 1_000_000 + i * T)
        t_before = buf.t
        ms_s, ms_s_local, launches_s = timed_steps(eng, buf, args.steps, torch, dist, world)
        sample.replay(buf.actions.cpu().numpy(), t_before, buf.t)
        check_s = sample.compare(eng, buf.last_obs(), torch, "steady steps")
        steady = {"value": n_total * args.steps / (ms_s / 1e3), "unit": UNIT, "ms_per_step": ms_s / args.steps,
                  "launch_ms": ms_s_local / args.steps, "gpu_launches": launches_s * world, "preroll_steps": (args.preroll // T) * T, "steps": args.steps,
                  "check": check_s,
                  "note": "same engine, same K timed nav3d_step launches, after an untimed pre-roll of fused random steps "
                          "(nav3d_rollout_random) that moves every env mid-episode"}
        if regime == "steady":
            steady["note"] += "; the main line already is a steady-state measurement"

    e2e_steps = max(3, min(args.e2e_steps, args.steps))
    sec, h2d, d2h, _, ceiling_gbs = time_e2e(eng, n_local, e2e_steps, torch, dist, world)
    e2e_value = n_total * e2e_steps / sec
    e2e_gbs = world * d2h * e2e_steps / sec / 1e9

    # roofline of the dominant kernel: measured on this rank's own stream with CUDA events
    peaks_file = ROOT / "MEASURED_PEAKS.json"
    if peaks_file.exists():
        peak, peak_src = float(json.loads(peaks_file.read_text())["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    else:
        peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
    balg = B_ALG.get(L, 334 + 64 + 64 + 12 * L + 2 + (6 * L + 1 + 7) // 8)
    if spec.get("simple"):
        balg = (6 * L + 7) * 4 + 14 + 64 + 2 * 6 * L + 2 + 4          # SURVEY §8d: 256 B at L = 4
    launch_ms = ms_local / args.steps
    achieved = balg * n_local / (launch_ms * 1e-3) / 1e9
    # DRAM bytes per launch from the committed ncu capture OF THE SAME REGIME (profiles/traffic.json), scaled to this shard
    traffic, traffic_src = None, None
    tf = ROOT / "profiles" / "traffic.json"
    if tf.exists():
        try:
            ent = json.loads(tf.read_text()).get(spec["name"], {}).get(regime)
            if ent:
                traffic = int(ent["dram_bytes_per_env_step"] * n_local)
                traffic_src = f"profiled, not measured in this run: {ent['source']}"
        except Exception:  # noqa: BLE001
            traffic = None
    kname = "simple_step_kernel" if spec.get("simple") else ("step_tpe_kernel" if eng.lanes_per_env == 1 else "step_call_kernel")
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "regime": regime,
                "kernel": kname + f"<lanes_per_env={eng.lanes_per_env}>",
                "algorithmic_bytes_per_env_step": balg, "env_steps_per_launch": n_local,
                "launch_ms": launch_ms, "peak_source": peak_src}
    if steady is not None:
        steady["roofline_frac"] = balg * n_local / (steady["launch_ms"] * 1e-3) / 1e9 / peak
        try:
            ent = json.loads(tf.read_text()).get(spec["name"], {}).get("steady")
            if ent:
                steady["traffic"] = int(ent["dram_bytes_per_env_step"] * n_local)
        except Exception:  # noqa: BLE001
            pass

    extra = {}
    cpu_baseline = None
    if not args.no_extras:
        try:
            extra["c5_train"] = time_training(torch, dist, world, rank, local_rank)
        except Exception as ex:  # noqa: BLE001
            extra["c5_train"] = {"error": repr(ex)}
    if rank == 0 and world == 1 and not args.no_extras:
        # secondary workloads, same timing method (short)
        del eng
        torch.cuda.empty_cache()
        for wl in ("c2", "c3"):
            if wl == spec["name"]:
                continue
            s2 = workload_spec(wl)
            r2 = load_rooms(s2)
            e2 = Engine(s2["envs_total"], r2, local_map_length=s2["L"], seed=2024, device=local_rank,
                        lanes_per_env=args.lanes)
            k2 = 2000
            m2, _, _ = time_steps(e2, s2["envs_total"], k2, 50, torch, dist, 1, act_rows=1024)
            extra[wl] = {"workload": s2["desc"], "value": s2["envs_total"] * k2 / (m2 / 1e3), "unit": UNIT,
                         "ms_per_step": m2 / k2, "steps": k2,
                         "roofline_frac": B_ALG[10] * s2["envs_total"] / (m2 / k2 * 1e-3) / 1e9 / peak}
            try:
                mg, kg = time_steps_graph(e2, s2["envs_total"], k2, torch)
                extra[wl]["cuda_graph"] = {"value": s2["envs_total"] * kg / (mg / 1e3), "ms_per_step": mg / kg, "steps": kg,
                                           "roofline_frac": B_ALG[10] * s2["envs_total"] / (mg / kg * 1e-3) / 1e9 / peak,
                                           "note": "50 nav3d_step launches captured per CUDA-graph replay"}
            except Exception as ex:  # noqa: BLE001
                extra[wl]["cuda_graph"] = {"error": str(ex)}
            del e2
            torch.cuda.empty_cache()
        # simpleEnv (envs/simpleEnv.py, the reference's older env variant): same timing method, 2^20 envs, L = 4
        try:
            from nav3d import _lib as nlib
            from nav3d.rooms import load_room_dir
            srooms = load_room_dir(ROOT / "rooms" / "P1_training", simple=True, sort=True)
            ns = 1 << 20
            es = Engine(ns, srooms, local_map_length=4, seed=2024, device=local_rank, lanes_per_env=args.lanes,
                        env_kind=nlib.ENV_SIMPLE)
            dsim = es.obs_dim
            g = torch.Generator(device=es.device).manual_seed(7)
            acts = torch.randint(0, 6, (320, ns), generator=g, device=es.device, dtype=torch.int64)   # one row per step
            sobs = torch.empty((4, ns, dsim), dtype=torch.float32, device=es.device)
            srew = torch.empty(ns, dtype=torch.float32, device=es.device)
            ste = torch.empty(ns, dtype=torch.uint8, device=es.device); strn = torch.empty(ns, dtype=torch.uint8, device=es.device)
            es.reset(sobs[0])
            for t in range(20):
                es.step(acts[t], sobs[t % 4], srew, ste, strn)
            torch.cuda.synchronize()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ks = 300
            ev0.record()
            for t in range(ks):
                es.step(acts[20 + t], sobs[t % 4], srew, ste, strn)
            ev1.record()
            torch.cuda.synchronize()
            msim = ev0.elapsed_time(ev1)
            extra["simple_env"] = {"workload": "2^20 simpleEnv envs (envs/simpleEnv.py), rooms/P1_training, L=4, random actions, auto-reset",
                                   "value": ns * ks / (msim / 1e3), "unit": UNIT, "ms_per_step": msim / ks, "steps": ks,
                                   "obs_dim": dsim, "lanes_per_env": es.lanes_per_env,
                                   "roofline_frac": 256 * ns / (msim / ks * 1e-3) / 1e9 / peak,
                                   "algorithmic_bytes_per_env_step": 256}
            del es, sobs, acts
            torch.cuda.empty_cache()
        except Exception as ex:  # noqa: BLE001
            extra["simple_env"] = {"error": repr(ex)}
        # fused random-action rollout (BASELINE.md §4 config 4: on-device Philox actions): one launch = T steps of every env,
        # EVERY observation, reward and done flag written ([T, N, 80] f32 = 10.7 GB at T = 32)
        try:
            s4 = workload_spec("c4")
            r4 = load_rooms(s4)
            e4 = Engine(s4["envs_total"], r4, local_map_length=10, seed=2024, device=local_rank, lanes_per_env=args.lanes)
            n4, T = s4["envs_total"], 32
            obs0 = e4.reset()
            obs_all = torch.empty((T, n4, 80), dtype=torch.float32, device=e4.device)
            rew = torch.empty((T, n4), dtype=torch.float32, device=e4.device)
            done = torch.empty((T, n4), dtype=torch.uint8, device=e4.device)
            smp = OracleSample(r4, 10, 2024, 0, n4)
            t0 = 0

            def fused(reps):
                nonlocal t0
                torch.cuda.synchronize()
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ev0.record()
                for _ in range(reps):
                    e4.rollout_random(T, t0, obs=obs_all, reward=rew, done=done)
                    smp.replay_random(T, t0)
                    t0 += T
                ev1.record()
                torch.cuda.synchronize()
                ms_r = ev0.elapsed_time(ev1)
                return {"value": n4 * T * reps / (ms_r / 1e3), "ms_per_env_step_batch": ms_r / (T * reps), "launches": reps,
                        "roofline_frac": B_ALG[10] * n4 * T * reps / (ms_r * 1e-3) / 1e9 / peak}

            fused(1)                                                   # warm-up launch (steps 0..31 of the episodes)
            cold = fused(6)
            cold["check"] = smp.compare(e4, obs_all[T - 1], torch, "fused rollout (cold)")
            for _ in range(576 // T):                                  # declared pre-roll: 576 more steps, last observation only
                e4.rollout_random(T, t0, obs_last=obs0)
                smp.replay_random(T, t0)
                t0 += T
            warm = fused(6)
            warm["check"] = smp.compare(e4, obs_all[T - 1], torch, "fused rollout (steady)")
            warm["preroll_steps"] = 576 + 7 * T
            ftraffic = {}
            try:
                ftraffic = json.loads(tf.read_text()).get("fused_rollout_full", {})
            except Exception:  # noqa: BLE001
                pass
            extra["fused_rollout_full"] = {
                "workload": "nav3d_rollout_random: 2^20 envs, P1_training, L=10, T=32 steps per launch, on-device Philox actions, "
                            "all T observations + rewards + done flags written (no work skipped)",
                "unit": UNIT, "T": T, "lanes_per_env": e4.lanes_per_env, "kernel": "rollout_tpe_kernel",
                "algorithmic_bytes_per_launch": B_ALG[10] * n4 * T, "cold": cold, "steady": warm,
                "dram_bytes_per_env_step_profiled": ftraffic}
            del e4, obs_all, rew, done
            torch.cuda.empty_cache()
        except Exception as ex:  # noqa: BLE001
            extra["fused_rollout_full"] = {"error": repr(ex)}
        # CPU baseline on this box's host cores (bounded sample): the reference itself when oracle/_ref travelled here
        cores = os.cpu_count() or 1
        per_worker = 100000 if cores >= 12 else 60000
        cb_rate, cb_wall, cb_one, cb_kind, cb_what = cpu_arm(spec, per_worker, cores, one_process_steps=10000)
        c_all = c_port_rate(rooms, L, 4096, 100, cores)
        c_one = c_port_rate(rooms, L, 512, 100, 1)
        cpu_baseline = {"value": cb_rate, "unit": UNIT, "cores": cores, "kind": cb_kind,
                        "sample": f"{cb_what}; {cores} worker processes x 1 env x {per_worker} random-action steps ({cb_wall:.1f} s)",
                        "one_process": cb_one,
                        "c_port": {"value": c_all, "cores": cores, "one_thread": c_one,
                                   "sample": "oracle/nav3d_oracle.c (C restatement, the parity checker): 4096 envs x 100 steps, pthreads"}}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": spec["scaling"], "vs_baseline": None,
            "dtype": "u8/u16 bit-packed state, f32 obs, f64 reward", "data": "synthetic",
            "config": {"workload": spec["desc"], "envs_total": n_total, "envs_per_gpu": n_local,
                       "lanes_per_env": roofline["kernel"], "local_map_length": L, "regime": regime,
                       "preroll_steps": 0, "action_rows": n_rows,
                       "l2": f"inputs larger than L2: {n_local * 21504 / 2**30:.1f} GiB of per-env knowledge per GPU vs 126 MB L2; no flush needed"
                             if n_local * 21504 > 4 * 126e6 else
                             "working set is L2-resident by design for this workload (not flushed: a trainer re-steps the same envs)",
                       "parallelism": f"env-sharded x{world}, no data-path collective"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": d2h * world,
                    "steps": e2e_steps, "api": "nav3d_step_host (pinned host buffers, per-step H2D actions + D2H obs/reward/flags)",
                    "numa": numa_note, "d2h_achieved_gbs": e2e_gbs, "host_ceiling_gbs": ceiling_gbs,
                    "host_ceiling_note": "aggregate of plain pinned device->host copies of the observation bytes, all ranks "
                                         "concurrently (the most this host side absorbs); d2h_achieved_gbs is what the e2e path moved"},
            "gpu_launches": launches * world,
            "roofline": roofline,
            "check": check,
            "steady": steady,
            "cpu_baseline": cpu_baseline,
            "clocks": clocks,
            "extra": extra,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
