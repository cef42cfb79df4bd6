#!/usr/bin/env python
"""Cost of the weighted room draw (nav3d_set_room_weights) on one GPU.  Three measurements, one JSON line:

  builder  : one nav3d_set_room_weights launch (device weights, no status read), CUDA events over --reps launches, at 25
             rooms (P2_training) and at 65 535 rooms;
  resets   : a workload that is nearly all resets: 2^20 envs in 25 copies of a 3x3x3 room with one free cell, where every
             step ends the episode (terminated and truncated) and auto-resets, nav3d_rollout_random T = 32 (obs_last only),
             with the uniform table and with a weighted 25-room table;
  default  : the default workload of bench.py (2^20 envs, P1_training, L = 10): per-step time of nav3d_step and of one
             T = 32 nav3d_rollout_random, in steady state after a 600-step fused pre-roll.
With --parent-tree DIR (a checkout of another commit with its library built), `resets` (uniform) and `default` run in child
processes that alternate between that tree's library and this one, --rounds times each, so their difference can be read
against the spread of the repeats.  Every child prints the card's name and power limit.
usage: python tools/room_weights_bench.py [--parent-tree DIR] [--rounds R]   -> one JSON line"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (s.strip() for s in q.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}


def events_ms(torch, fn, reps):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / reps


def tiny_rooms(n):
    import numpy as np
    from nav3d.rooms import rooms_from_grids
    g = np.full((3, 3, 3), -2, np.int8)
    g[1, 1, 1] = 0
    return rooms_from_grids([g] * n)


def child(tree: Path, what: str, weighted: bool):
    sys.path.insert(0, str(tree))
    import _nav3d_path  # noqa: F401  (the package of `tree`)
    import numpy as np
    import torch
    from nav3d import Engine
    from nav3d.rooms import load_room_dir
    n, T = 1 << 20, 32
    out = {"tree": str(tree), "card": card()}
    if what == "resets":
        eng = Engine(n, tiny_rooms(25), local_map_length=10, seed=1)
        if weighted:
            eng.set_room_weights(np.random.default_rng(0).random(25).astype(np.float32) * (np.arange(25) % 5 != 0))
        obs = eng.new_obs()
        eng.reset(obs)
        t0 = [0]

        def roll():
            eng.rollout_random(T, t0[0], obs_last=obs)
            t0[0] += T
        ms = events_ms(torch, roll, 20)
        out.update(ms_per_rollout=ms, ns_per_env_step=ms * 1e6 / (n * T), resets_per_rollout=n * T)
    else:
        eng = Engine(n, load_room_dir(ROOT / "rooms" / "P1_training", sort=True), local_map_length=10, seed=1)
        obs = eng.reset()
        eng.rollout_random(600, 1_000_000, obs_last=obs)
        dev = eng.device
        acts = [torch.randint(0, 6, (n,), generator=torch.Generator().manual_seed(i)).to(dev) for i in range(8)]
        rew, te, tr = torch.zeros(n, device=dev), torch.zeros(n, dtype=torch.uint8, device=dev), \
            torch.zeros(n, dtype=torch.uint8, device=dev)
        i = [0]

        def step():
            eng.step(acts[i[0] % 8], obs, rew, te, tr)
            i[0] += 1
        t0 = [2_000_000]

        def roll():
            eng.rollout_random(T, t0[0], obs_last=obs)
            t0[0] += T
        out.update(ms_per_step=events_ms(torch, step, 400), ms_per_rollout_T32=events_ms(torch, roll, 20))
    print(json.dumps(out), flush=True)


def run_child(tree: Path, what: str, weighted: bool = False):
    cmd = [sys.executable, str(Path(__file__).resolve()), "--child", what, "--tree", str(tree)] + (["--weighted"] if weighted else [])
    r = subprocess.run(cmd, capture_output=True, text=True, check=True)
    return json.loads(r.stdout.strip().splitlines()[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-tree", type=Path)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--child", choices=["resets", "default"])
    ap.add_argument("--tree", type=Path, default=ROOT)
    ap.add_argument("--weighted", action="store_true")
    args = ap.parse_args()
    if args.child:
        return child(args.tree, args.child, args.weighted)
    sys.path.insert(0, str(ROOT))
    import _nav3d_path  # noqa: F401
    import numpy as np
    import torch
    from nav3d import Engine
    from nav3d.rooms import load_room_dir
    res = {"tool": "room_weights_bench", "card": card(), "builder": {}}
    for label, rooms in (("25 rooms (P2_training)", load_room_dir(ROOT / "rooms" / "P2_training", sort=True)),
                         ("65535 rooms", tiny_rooms(65535))):
        eng = Engine(8, rooms, local_map_length=10)
        w = torch.rand(len(rooms), generator=torch.Generator().manual_seed(0)).to(eng.device)
        res["builder"][label] = {"us_per_launch": 1e3 * events_ms(torch, lambda: eng.set_room_weights(w, check=False),
                                                                  args.reps)}
        del eng
    res["resets"] = {"weighted_25": run_child(ROOT, "resets", True), "uniform": [], "uniform_parent": []}
    res["default"] = {"new": [], "parent": []}
    for _ in range(args.rounds):
        for key, tree in (("parent", args.parent_tree), ("new", ROOT)):
            if tree is None:
                continue
            res["resets"]["uniform" if key == "new" else "uniform_parent"].append(run_child(tree, "resets"))
            res["default"][key].append(run_child(tree, "default"))
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
