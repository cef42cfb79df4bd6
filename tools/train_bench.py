#!/usr/bin/env python
"""Throughput of the LSTM-PPO loop on the GPU-resident env: time split between rollout collection and the PPO update.
usage: python tools/train_bench.py [--envs N --n-steps T --batch-envs B --iters K --epochs E]"""
import argparse
import json
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import _nav3d_path  # noqa: E402,F401


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--n-steps", type=int, default=128)
    ap.add_argument("--batch-envs", type=int, default=512)
    ap.add_argument("--iters", type=int, default=4)
    ap.add_argument("--epochs", type=int, default=10)
    ap.add_argument("--rooms", default="P1_training")
    ap.add_argument("--two-streams", type=int, default=1)
    ap.add_argument("--curriculum", type=int, default=0, help="1: attach a nav3d.curriculum.RoomCurriculum to the env")
    args = ap.parse_args()
    import torch
    from nav3d import BatchedCubicEnv
    from nav3d.ppo import RecurrentPPO
    env = BatchedCubicEnv(ROOT / "rooms" / args.rooms, num_envs=args.envs, local_map_length=10, seed=42, sort_rooms=True)
    m = RecurrentPPO(env, policy_kwargs=dict(net_arch=dict(pi=[256, 256, 128], vf=[256, 256, 128]), lstm_hidden_size=256,
                                             n_lstm_layers=1),
                     learning_rate=3e-4, n_steps=args.n_steps, batch_size=args.batch_envs * args.n_steps, n_epochs=args.epochs,
                     gamma=0.99, gae_lambda=0.95, ent_coef=0.01, vf_coef=0.5, clip_range=0.2, seed=0)
    if args.curriculum:
        from nav3d.curriculum import RoomCurriculum
        m.curriculum = RoomCurriculum(env)
    m.policy.two_streams = bool(args.two_streams)
    for _ in range(2):                                   # warm-up: eager rollout, then the rollout's CUDA-graph capture
        m.collect_rollouts(); m.train()
    torch.cuda.synchronize()
    t_roll = t_train = 0.0
    for _ in range(args.iters):
        t0 = time.perf_counter(); m.collect_rollouts(); torch.cuda.synchronize(); t1 = time.perf_counter()
        st = m.train(); torch.cuda.synchronize(); t2 = time.perf_counter()
        t_roll += t1 - t0; t_train += t2 - t1
    steps = args.iters * args.n_steps * args.envs
    print(json.dumps(dict(two_streams=args.two_streams, curriculum=args.curriculum, envs=args.envs, n_steps=args.n_steps, batch_envs=args.batch_envs, epochs=args.epochs,
                          rollout_steps_per_s=steps / t_roll, train_steps_per_s=steps / t_train,
                          total_steps_per_s=steps / (t_roll + t_train), rollout_ms_per_step=1e3 * t_roll / (args.iters * args.n_steps),
                          minibatches=st["minibatches"], reward_mean=st["rollout_reward_mean"])))


if __name__ == "__main__":
    main()
