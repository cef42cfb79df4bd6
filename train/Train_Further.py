"""Continue training saved LSTM-PPO models for one more phase (P2) on the GPU-resident CubicEnv.

Drop-in for the reference's ``train/Train_Further.py``: every ``*.zip`` in ``LOAD_DIR`` is loaded (network, optimiser and
step counter included), its ray length is parsed from the ``_view<N>.zip`` suffix, training continues for
``STEPS_PHASE["P2_small"]`` steps in ten segments, and after each segment the model is saved as ``<name>_P2.zip_i`` under
``SAVE_DIR`` — the reference's file names, odd suffix included.

    python -m train.Train_Further [--load-dir D --save-dir D --steps N --num-envs N]"""
import argparse
import glob
import os
import random
import sys
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import _nav3d_path  # noqa: E402,F401

from nav3d.evaluation import EvalCallback  # noqa: E402
from nav3d.experiment import (BASE_SEED, continued_name, dist_setup, eval_every_calls, make_vec_env,  # noqa: E402
                              parse_view_suffix, split_segments)
from nav3d.curriculum import RoomCurriculum  # noqa: E402
from nav3d.ppo import RecurrentPPO  # noqa: E402

random.seed(BASE_SEED)
np.random.seed(BASE_SEED)
NUM_ENVS = 8
CRASH_PENALTIES = [-2.0]

LOAD_DIR = "./exp3_architectures/best_P1_empty_r10_cp-2.0"
SAVE_DIR = "./exp3_architectures/P2"
EVAL_FREQ = 100_000

PHASES = [("P2_small", "./rooms/P2_training", "./rooms/P2_evaluate")]
STEPS_PHASE = {"P2_small": 20_000_000}


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--load-dir", default=LOAD_DIR)
    ap.add_argument("--save-dir", default=SAVE_DIR)
    ap.add_argument("--steps", type=int, default=0)
    ap.add_argument("--num-envs", type=int, default=NUM_ENVS)
    ap.add_argument("--eval-freq", type=int, default=EVAL_FREQ)
    ap.add_argument("--curriculum", action="store_true",
                    help="draw the training rooms from learning-progress weights (nav3d.curriculum.RoomCurriculum), starting "
                         "afresh on this phase's rooms; evaluation is unchanged")
    args = ap.parse_args(argv)
    rank, world, local_rank = dist_setup()
    phase_name, train_path, eval_path = PHASES[0]
    if not os.path.exists(train_path) or not os.path.exists(eval_path):
        print("Error: Phase 2 training or evaluation directory not found.")
        return 1
    best_model_dir = os.path.join(args.save_dir, "best_exp3_P2")
    if rank == 0:
        os.makedirs(best_model_dir, exist_ok=True)
    model_files = glob.glob(os.path.join(args.load_dir, "*.zip"))
    if not model_files:
        print(f"No .zip models found in {args.load_dir}. Exiting.")
        return 1
    print(f"Found {len(model_files)} models to continue training.")
    for model_path in model_files:
        model_filename = os.path.basename(model_path)
        print(f"\n{'=' * 40}\nProcessing model: {model_filename}\n{'=' * 40}")
        ray_len = parse_view_suffix(model_filename)
        if ray_len is None:
            print(f"Warning: Could not parse 'ray_len' from filename: {model_filename}. Skipping this model.")
            continue
        steps_this_phase = args.steps or STEPS_PHASE[phase_name]
        eval_env = make_vec_env(eval_path, ray_len, NUM_ENVS, NUM_ENVS, rank=rank, device=local_rank)
        train_env = make_vec_env(train_path, ray_len, args.num_envs, 0, rank=rank, device=local_rank)
        model = RecurrentPPO.load(model_path, env=train_env, verbose=1)
        print(f"Model loaded ({model.num_timesteps} steps so far). Continuing training on {phase_name}.")
        if args.curriculum:
            model.curriculum = RoomCurriculum(train_env)
        for i, seg_steps in enumerate(split_segments(steps_this_phase)):
            print(f"\n--- Training {phase_name} segment {i + 1}/10 ({seg_steps} steps) ---")
            eval_callback = EvalCallback(eval_env=eval_env, best_model_save_path=best_model_dir, log_path=best_model_dir,
                                         eval_freq=eval_every_calls(args.eval_freq, args.num_envs * world),
                                         n_eval_episodes=10, deterministic=True, render=False)
            model.learn(total_timesteps=seg_steps, reset_num_timesteps=False, callback=eval_callback)
            save_path = os.path.join(args.save_dir, continued_name(model_filename))
            model.save(save_path)
            print(f"Checkpoint saved to: {save_path}")
        print(f"Finished training for {model_filename}.")
        train_env.close()
        eval_env.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
