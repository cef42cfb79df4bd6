#!/usr/bin/env python
"""Cost of the per-room episode statistics (nav3d_room_stats) on one GPU, against the index_add_ recipe the project's
INTEGRATION.md used before (two index_add_ over all T x N rows into R + 1 float bins: finished episodes and successes).

Workloads, each at 2^20 envs x T = 32 (the bench.py shape):
  a) rollout : flags and episodes of a real nav3d_rollout_actions on P1_training, after a 600-step pre-roll;
  b) one_room: every row done, all in room 0 (of P1_training's rooms);
  c) random  : 65 535 rooms, every row done, rooms drawn uniformly.
For each the kernel and the recipe are timed alternately with CUDA events, --reps calls per round and --rounds rounds,
twice: with the same buffers every call (the 64 MiB of flags can stay in the 126 MB L2) and with a 512 MiB scratch buffer
written between calls (not timed), which evicts them.  Bytes the kernel must read = 2 T N (flags) + 32 per done row; the
rate is stated against 7.7 TB/s of HBM3e.  The card's name and power limit are read in the same run.
usage: python tools/room_stats_bench.py [--reps 50] [--rounds 3]   -> one JSON line"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import _nav3d_path  # noqa: E402,F401

HBM_BPS = 7.7e12


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (s.strip() for s in q.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    import numpy as np
    import torch
    from nav3d import Engine
    from nav3d.rooms import load_room_dir, rooms_from_grids
    if not torch.cuda.is_available():
        raise SystemExit("room_stats_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    N, T = 1 << 20, 32
    g = torch.Generator(dev).manual_seed(0)
    p1 = load_room_dir(ROOT / "rooms" / "P1_training", sort=True)
    eng_p1 = Engine(N, p1, local_map_length=10, seed=1)
    obs = eng_p1.reset()
    for k in range(600 // T):
        eng_p1.rollout_random(T, k * T, obs_last=obs)
    te = torch.zeros((T, N), dtype=torch.uint8, device=dev)
    tr = torch.zeros_like(te)
    ep = torch.zeros((T, N, 8), dtype=torch.int32, device=dev)
    acts = torch.randint(0, 6, (T, N), dtype=torch.uint8, device=dev, generator=g)
    eng_p1.rollout_actions(acts, obs_last=obs, terminated=te, truncated=tr, episodes=ep)

    def synthetic(R, room):
        e = torch.randint(0, 1000, (T, N, 8), dtype=torch.int32, device=dev, generator=g)
        e[..., 0] = (torch.randn((T, N), device=dev, generator=g) * 300).view(torch.int32)
        e[..., 5] = room if room is not None else torch.randint(0, R, (T, N), dtype=torch.int32, device=dev, generator=g)
        return torch.ones((T, N), dtype=torch.uint8, device=dev), torch.zeros((T, N), dtype=torch.uint8, device=dev), e

    cell = np.full((3, 3, 3), -2, np.int8)
    cell[1, 1, 1] = 0
    eng_r = Engine(N, rooms_from_grids([cell] * 65535), local_map_length=4)
    workloads = {"rollout": (eng_p1, te, tr, ep), "one_room": (eng_p1, *synthetic(len(p1), 0)),
                 "random": (eng_r, *synthetic(65535, None))}
    scratch = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    out = {"card": card(), "shape": {"n_envs": N, "T": T}, "reps": args.reps, "rounds": args.rounds, "workloads": {}}
    for name, (eng, t, r, e) in workloads.items():
        R = len(eng.rooms)
        acc = torch.zeros((R, 8), dtype=torch.int64, device=dev)
        ends = torch.zeros(R + 1, device=dev)
        wins = torch.zeros(R + 1, device=dev)

        def kernel():
            eng.room_stats(t, r, e, out=acc)

        def recipe():
            done = (t | r).bool()
            room = torch.where(done, e[..., 5], R).long().flatten()
            ends.index_add_(0, room, done.flatten().float())
            wins.index_add_(0, room, e[..., 6].flatten().float() * done.flatten())

        n_done = int((t | r).ne(0).sum())
        bytes_needed = 2 * T * N + 32 * n_done
        res = {"rooms": R, "done_rows": n_done, "bytes_needed": bytes_needed}
        acc.zero_()
        kernel()
        assert int(acc[:, 0].sum()) == n_done, name           # (the recipe's float32 bins stop counting at 2^24)
        for mode in ("warm", "cold"):
            times = {"kernel": [], "index_add": []}
            for _ in range(args.rounds):
                for which, fn in (("kernel", kernel), ("index_add", recipe)):
                    fn()
                    tot = 0.0
                    for _ in range(args.reps):
                        if mode == "cold":
                            scratch.fill_(1)
                        s, f = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        s.record(); fn(); f.record()
                        f.synchronize()
                        tot += s.elapsed_time(f)
                    times[which].append(1e3 * tot / args.reps)
            k_us = min(times["kernel"])
            res[mode] = {"kernel_us": [round(x, 2) for x in times["kernel"]],
                         "index_add_us": [round(x, 2) for x in times["index_add"]],
                         "kernel_bytes_per_s": bytes_needed / (k_us * 1e-6),
                         "kernel_share_of_7.7TBps": bytes_needed / (k_us * 1e-6) / HBM_BPS,
                         "speedup_vs_index_add": min(times["index_add"]) / k_us}
        res["flags_note"] = ("warm: the same 64 MiB of flags every call, which fit the 126 MB L2; cold: a 512 MiB write "
                             "between calls evicts them")
        out["workloads"][name] = res
    print(json.dumps(out))


if __name__ == "__main__":
    main()
