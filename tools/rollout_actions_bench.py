#!/usr/bin/env python
"""Fused rollout with caller-supplied actions (nav3d_rollout_actions) against the fused Philox rollout
(nav3d_rollout_random) and T nav3d_step launches with the same actions.  One GPU, 2^20 envs of P1_training, L = 10, T = 32,
every observation written; the actions are uniform random, generated on the device from a fixed seed before timing.

The three arms alternate, one rollout of T steps each, in two regimes: cold (every env reset before each repetition; the
reset is not timed) and steady (after a 600-step fused pre-roll; the arms then continue the same episodes).  Each
repetition draws fresh action rows (untimed) for arms 1 and 3: replaying one fixed block would let every env repeat a
32-step pattern, drift into a wall and keep bumping there, which makes the steps cheaper (DESIGN §6).  CUDA events
around each repetition, at least --seconds of timed work per arm.  Rates: env-steps/s and the fraction of the 6 452.8 GB/s
copy peak at DESIGN §5's 592 algorithmic bytes per env-step (of which 8 are the int64 action nav3d_step reads; this call
reads one byte).  Before timing, arms 1 and 3 are run from the same saved state and their outputs compared bit for bit.
usage: python tools/rollout_actions_bench.py [--envs N --T T --seconds S]   -> one JSON line"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import _nav3d_path  # noqa: E402,F401

BYTES_PER_ENV_STEP = 592
PEAK_GBS = 6452.8


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
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--T", type=int, default=32)
    ap.add_argument("--seconds", type=float, default=0.5, help="least timed work per arm and regime")
    ap.add_argument("--preroll", type=int, default=600)
    args = ap.parse_args()
    import torch
    from nav3d import Engine
    from nav3d.rooms import load_room_dir
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    rooms = load_room_dir(ROOT / "rooms" / "P1_training", sort=True)
    n, T = args.envs, args.T
    eng = Engine(n, rooms, local_map_length=10, seed=2024)
    dev = eng.device
    gen = torch.Generator(device=dev).manual_seed(7)
    acts = torch.randint(0, 6, (T, n), generator=gen, device=dev, dtype=torch.uint8)
    acts64 = acts.long()

    def new_actions():
        torch.randint(0, 6, (T, n), generator=gen, device=dev, dtype=torch.uint8, out=acts)
        acts64.copy_(acts)
    obs = torch.empty((T, n, 80), device=dev)
    rew = torch.empty((T, n), device=dev)
    te = torch.empty((T, n), dtype=torch.uint8, device=dev)
    tr = torch.empty((T, n), dtype=torch.uint8, device=dev)
    done = torch.empty((T, n), dtype=torch.uint8, device=dev)
    cur = eng.reset()
    t0 = [0]

    def arm_actions():
        eng.rollout_actions(acts, obs=obs, reward=rew, terminated=te, truncated=tr)

    def arm_random():
        eng.rollout_random(T, t0[0], obs=obs, reward=rew, done=done)
        t0[0] += T

    def arm_steps():
        for t in range(T):
            eng.step(acts64[t], obs[t], rew[t], te[t], tr[t])

    # arms 1 and 3 from the same state: identical outputs and final records
    ids = torch.arange(n, dtype=torch.int32, device=dev)
    for _ in range(3):
        arm_steps()
    blobs = eng.save_envs(ids, obs[-1].contiguous())
    arm_actions()
    got = [x.clone() for x in (obs, rew, te, tr)] + [eng.get_state()]
    eng.load_envs(ids, blobs, cur, check=False)
    arm_steps()
    want = [obs, rew, te, tr, eng.get_state()]
    identical = all(torch.equal(a.view(torch.uint8), b.view(torch.uint8)) for a, b in zip(got, want))
    del blobs, got, want
    torch.cuda.empty_cache()

    arms = {"rollout_actions": arm_actions, "rollout_random": arm_random, "step_x_T": arm_steps}
    out = {"card": card(), "envs": n, "T": T, "outputs": "obs [T,N,80] + reward + flags", "arms_1_3_identical": identical}
    for f in arms.values():                      # warm-up of every arm
        f()
    for regime in ("cold", "steady"):
        if regime == "steady":
            eng.reset(cur)
            for _ in range(args.preroll // T):
                eng.rollout_random(T, t0[0], obs_last=cur)
                t0[0] += T
        ms = {k: 0.0 for k in arms}
        reps = 0
        while min(ms.values()) < args.seconds * 1e3:
            new_actions()
            evs = []
            for name, f in arms.items():
                if regime == "cold":
                    eng.reset(cur)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                f()
                e1.record()
                evs.append((name, e0, e1))
            torch.cuda.synchronize()
            for name, e0, e1 in evs:
                ms[name] += e0.elapsed_time(e1)
            reps += 1
        res = {"repetitions": reps}
        for name, m in ms.items():
            us = m * 1e3 / (reps * T)
            rate = n / (us * 1e-6)
            res[name] = {"us_per_step": round(us, 1), "env_steps_per_s": float(f"{rate:.4g}"),
                         "frac_of_peak": round(BYTES_PER_ENV_STEP * rate / (PEAK_GBS * 1e9), 3)}
        out[regime] = res
    out["card_after"] = card()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
