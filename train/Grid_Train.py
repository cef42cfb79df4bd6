"""Multi-phase LSTM-PPO training on the GPU-resident CubicEnv, with a checkpoint after every tenth of a phase.

Drop-in for the reference's ``train/Grid_Train.py`` (same experiment grid, phases, hyper-parameters, seeding, evaluation
cadence and checkpoint names), with ``SubprocVecEnv`` + sb3-contrib replaced by ``nav3d.BatchedCubicEnv`` +
``nav3d.ppo.RecurrentPPO``:

    python -m train.Grid_Train                      # the reference's constants (8 envs, n_steps 2048, batch 64)
    python -m train.Grid_Train --native             # B200-sized rollouts: 1024 envs x 128 steps, 64 Ki-transition minibatches
    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 -m train.Grid_Train --native   # data parallel

Deviations, all deliberate: ``STEPS_PHASE`` has an entry for every phase (the reference's only active phase has none and
raises KeyError, Grid_Train.py:53-61/:176); ``check_env`` (an SB3 utility) is replaced by a one-step smoke check."""
import argparse
import os
import random
import sys
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import _nav3d_path  # noqa: E402,F401

from nav3d.evaluation import EvalCallback  # noqa: E402
from nav3d.experiment import (BASE_SEED, arch_string, checkpoint_name, dist_setup, eval_every_calls, lstm_string,  # noqa: E402
                              make_vec_env, split_segments)
from nav3d.curriculum import RoomCurriculum  # noqa: E402
from nav3d.ppo import RecurrentPPO  # noqa: E402

random.seed(BASE_SEED)
np.random.seed(BASE_SEED)
NUM_ENVS = 8
LOCAL_MAP_LENGTHS = [10]            # ray length of GridAgent._sense_direction
CRASH_PENALTIES = [-2.0]            # never forwarded to the env, as in the reference (GridEnv drops it)

SAVE_DIR = "./exp3_architectures"
EVAL_FREQ = 100_000

PHASES = [
    ("P1_empty", "./rooms/P1_training", "./rooms/P1_evaluate"),
    # ("P2_small", "./rooms/P2_training", "./rooms/P2_evaluate"),
    # ("P3_large", "./rooms/P3_training", "./rooms/P3_evaluate"),
]
STEPS_PHASE = {"P1_empty": 20_000_000, "P2_small": 20_000_000, "P3_large": 2_000_000}

architectures = [dict(pi=[256, 256, 128], vf=[256, 256, 128])]
lstm_sizes = [dict(lstm_hidden_size=256, n_lstm_layers=1)]
ppo_hparam_sets = [dict(learning_rate=3e-4, n_steps=2048, batch_size=64, gamma=0.99, gae_lambda=0.95, ent_coef=0.01,
                        vf_coef=0.5, clip_range=0.2, n_epochs=10)]
NATIVE_OVERRIDES = dict(n_steps=128, batch_size=512 * 128)      # --native: 512 envs x 128 steps per minibatch
NATIVE_NUM_ENVS = 1024              # the shape of profiles/train_demo_r01 (100 % finished on P1_evaluate after 72 M steps)
NATIVE_EVAL_FREQ = 5_000_000        # at ~1e6 steps/s an evaluation every 100 k steps would dominate the run


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--native", action="store_true", help="B200-sized rollout/minibatch shape instead of the reference's")
    ap.add_argument("--num-envs", type=int, default=0, help="envs per GPU (default 8, or 1024 with --native)")
    ap.add_argument("--steps", type=int, default=0, help="override the steps of every phase")
    ap.add_argument("--save-dir", default=SAVE_DIR)
    ap.add_argument("--eval-freq", type=int, default=0, help="steps between evaluations (default 100000; 5000000 with --native)")
    ap.add_argument("--phases", default="", help="comma-separated phase names to run (default: the PHASES list)")
    ap.add_argument("--curriculum", action="store_true",
                    help="draw each phase's training rooms from learning-progress weights (nav3d.curriculum.RoomCurriculum) "
                         "instead of uniformly; evaluation is unchanged")
    args = ap.parse_args(argv)
    rank, world, local_rank = dist_setup()
    num_envs = args.num_envs or (NATIVE_NUM_ENVS if args.native else NUM_ENVS)
    eval_freq = args.eval_freq or (NATIVE_EVAL_FREQ if args.native else EVAL_FREQ)
    save_dir = args.save_dir
    best_model_dir = os.path.join(save_dir, "best_exp3_P1")
    if rank == 0:
        os.makedirs(best_model_dir, exist_ok=True)
    all_phases = {"P1_empty": ("./rooms/P1_training", "./rooms/P1_evaluate"),
                  "P2_small": ("./rooms/P2_training", "./rooms/P2_evaluate"),
                  "P3_large": ("./rooms/P3_training", "./rooms/P3_evaluate")}
    phases = PHASES if not args.phases else [(p, *all_phases[p]) for p in args.phases.split(",")]

    # the reference runs SB3's check_env here; the equivalent smoke check: one reset and one step of the first phase's env
    probe = make_vec_env(phases[0][1], LOCAL_MAP_LENGTHS[0], 2, 0, rank=rank, device=local_rank)
    obs = probe.reset()
    assert tuple(obs.shape) == (2, 80) and bool(((obs >= -1) & (obs <= 1)).all())
    probe.step(np.zeros(2, dtype=np.int64))
    probe.close()
    if rank == 0:
        print("Environment check passed.")

    for ray_len in LOCAL_MAP_LENGTHS:
        for hp_i, ppo_hp in enumerate(ppo_hparam_sets):
            hp = dict(ppo_hp, **(NATIVE_OVERRIDES if args.native else {}))
            for arch in architectures:
                arch_str = arch_string(arch)
                for lstm_kwargs in lstm_sizes:
                    lstm_str = lstm_string(lstm_kwargs)
                    base_id = f"r{ray_len}_arch{arch_str}_lstm{lstm_str}"
                    model = None
                    cumulative_steps_total = 0
                    for phase_name, train_path, eval_path in phases:
                        if rank == 0:
                            print(f"\n{'=' * 20}\nSTARTING PHASE: {phase_name} for {base_id}\n{'=' * 20}")
                        steps_this_phase = args.steps or STEPS_PHASE[phase_name]
                        if steps_this_phase <= 0:
                            print(f"Skipping phase {phase_name} as it has 0 steps.")
                            continue
                        eval_env = make_vec_env(eval_path, ray_len, NUM_ENVS, NUM_ENVS, rank=rank, device=local_rank)
                        train_env = make_vec_env(train_path, ray_len, num_envs, 0, rank=rank, device=local_rank)
                        segments = split_segments(steps_this_phase)
                        if model is None:
                            if rank == 0:
                                print("Instantiating new model.")
                            model = RecurrentPPO(train_env, policy="MlpLstmPolicy", verbose=1,
                                                 policy_kwargs=dict(net_arch=arch, **lstm_kwargs), seed=BASE_SEED, **hp)
                        else:
                            if rank == 0:
                                print(f"Continuing training on {phase_name}. Setting new environment.")
                            model.set_env(train_env)
                        if args.curriculum:
                            model.curriculum = RoomCurriculum(train_env)
                        for i, seg_steps in enumerate(segments):
                            cumulative_steps_total += seg_steps
                            if rank == 0:
                                print(f"\n--- Training {phase_name} segment {i + 1}/{len(segments)} ({seg_steps} steps) ---")
                                print(f"--- Cumulative steps for this model: {cumulative_steps_total} ---")
                            eval_callback = EvalCallback(eval_env=eval_env, best_model_save_path=best_model_dir,
                                                         log_path=best_model_dir,
                                                         eval_freq=eval_every_calls(eval_freq, num_envs * world),
                                                         n_eval_episodes=10, deterministic=True, render=False)
                            model.learn(total_timesteps=seg_steps, reset_num_timesteps=False, callback=eval_callback)
                            save_path = os.path.join(save_dir, checkpoint_name(hp_i + 1, arch_str, lstm_str,
                                                                               cumulative_steps_total, ray_len))
                            model.save(save_path)
                            if rank == 0:
                                print(f"Checkpoint saved to: {save_path}")
                        train_env.close()
                        eval_env.close()
    if rank == 0:
        print("\nAll incremental exploration experiments with checkpoints completed.")


if __name__ == "__main__":
    main()
