#!/usr/bin/env python
"""Bandwidth of the env-state blob calls (nav3d_save_envs / nav3d_load_envs) against a plain device-to-device copy of the
same size (Tensor.copy_, a cudaMemcpyAsync), on one GPU.

Two engines: P1_training at 2^20 envs and the 42 rooms of P2 + P3 training at 65 536 envs, L = 10, each after a 200-step
random-action pre-roll (nav3d_rollout_random).  For each, save and load of 2^14 and 2^17 random distinct envs (of the
65 536-env engine: 2^14 and all of them) are timed
with CUDA events, after a warm-up, over as many back-to-back calls as fill at least --min-seconds.  The same env set is
saved (loaded) on every call.

Bytes moved = what the call must read plus what it must write: per env, the header and record (64 B), the observation row
and the live part of the knowledge block (K of the env's room + its W*D*H overflow bytes), once read and once written.
The copy ceiling moves the same number of bytes (half read, half written).  The card name and power limit are read in
the same process.  Prints one JSON line and, with --out-dir, writes it to DIR/env_state_bench.json.
usage: python tools/env_state_bench.py [--out-dir DIR] [--min-seconds 0.5]"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import _nav3d_path  # noqa: E402,F401


def card():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        out.update({"smi_name": q[0], "power_limit": q[1], "sm_max_clock": q[2]})
    except Exception as ex:  # noqa: BLE001
        out["power_limit"] = f"unavailable ({ex})"
    return out


def live_bytes(eng, envs):
    """Bytes of the live part of each listed env's block (K of its room + the room's overflow bytes), from nav3d_get_state."""
    rooms = eng.get_state()[:, 13].cpu().numpy()[envs]
    per_room = []
    for (w, d, h) in eng.room_dims:
        k = ((w + 6) // 4) * ((d + 6) // 4) * ((h + 5) // 6) * 64        # nav3d_core.cuh k_bytes of the bordered volume
        per_room.append(k + w * d * h)
    return np.asarray(per_room, np.int64)[rooms]


def timed(fn, min_seconds):
    import torch
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 4
    while True:
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if ms >= min_seconds * 1e3:
            return ms / reps, reps
        reps = max(reps * 2, int(reps * min_seconds * 1.2e3 / max(ms, 1e-3)))


def bench_engine(name, rooms, n_envs, sizes, min_seconds, seed):
    import torch
    from nav3d import Engine
    eng = Engine(n_envs, rooms, local_map_length=10, seed=seed)
    dev = eng.device
    obs = eng.reset()
    eng.rollout_random(200, 0, obs_last=obs)
    torch.cuda.synchronize()
    B = eng.env_state_bytes
    rng = np.random.default_rng(seed)
    res = {"rooms": name, "envs": n_envs, "n_rooms": len(rooms), "blob_bytes": B, "runs": []}
    for n in sizes:
        ids_h = rng.choice(n_envs, n, replace=False).astype(np.int32)
        ids = torch.as_tensor(ids_h, device=dev)
        blobs = torch.empty((n, B), dtype=torch.uint8, device=dev)
        live = live_bytes(eng, ids_h)
        moved = int(2 * (live.sum() + n * (64 + 320)))            # read + written
        save_ms, save_reps = timed(lambda: eng.save_envs(ids, obs, out=blobs), min_seconds)
        load_ms, load_reps = timed(lambda: eng.load_envs(ids, blobs, obs, check=False), min_seconds)
        half = moved // 2
        src = torch.empty(half, dtype=torch.uint8, device=dev)
        dst = torch.empty_like(src)
        src.fill_(1)
        copy_ms, copy_reps = timed(lambda: dst.copy_(src), min_seconds)
        del src, dst
        gbs = lambda ms: moved / (ms * 1e-3) / 1e9  # noqa: E731
        res["runs"].append({
            "n": n, "bytes_moved": moved, "live_bytes_per_env_mean": float(live.mean()),
            "full_blob_bytes": n * B,
            "save_us": save_ms * 1e3, "save_GBps": gbs(save_ms), "save_reps": save_reps,
            "load_us": load_ms * 1e3, "load_GBps": gbs(load_ms), "load_reps": load_reps,
            "d2d_copy_us": copy_ms * 1e3, "d2d_copy_GBps": gbs(copy_ms), "copy_reps": copy_reps,
            "save_vs_copy": copy_ms / save_ms, "load_vs_copy": copy_ms / load_ms})
        del blobs
        torch.cuda.synchronize()
    eng.close()
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out-dir", default=None)
    ap.add_argument("--min-seconds", type=float, default=0.5)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("env_state_bench.py needs a CUDA device; there is nothing to measure without one")
    from nav3d.rooms import load_room_dir
    p1 = load_room_dir(ROOT / "rooms" / "P1_training", sort=True)
    p23 = load_room_dir(ROOT / "rooms" / "P2_training", sort=True) + load_room_dir(ROOT / "rooms" / "P3_training", sort=True)
    out = {"tool": "env_state_bench", "card": card(), "L": 10, "preroll_steps": 200, "min_seconds": args.min_seconds,
           "results": [bench_engine("P1_training", p1, 1 << 20, [1 << 14, 1 << 17], args.min_seconds, 1),
                       bench_engine("P2_training+P3_training", p23, 1 << 16, [1 << 14, 1 << 16], args.min_seconds, 2)]}
    line = json.dumps(out)
    print(line)
    if args.out_dir:
        d = Path(args.out_dir)
        d.mkdir(parents=True, exist_ok=True)
        (d / "env_state_bench.json").write_text(line + "\n")


if __name__ == "__main__":
    main()
