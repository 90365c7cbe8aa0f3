"""Reference side: turn the VecNormalize `.pkl` that the reference's CheckpointCallback writes (train_hover.py:17-31) into the
`.npz` that `eval_hover_b200.py --vecnormalize` and `sac.load_vecnormalize` read -- the keys `ppo.export_sb3_zip` uses for
`vecnormalize.npz` (obs_rms.mean / .var / .count, ret_rms.*, clip_obs, clip_reward, gamma, epsilon, norm_obs, norm_reward).

    python tools/sb3_vecnormalize_to_npz.py hover_vecnormalize.pkl out.npz [--task hover|yaw]

It loads the pickle with stable-baselines3's own `VecNormalize.load`, so it runs only where SB3 and gymnasium are installed
(the reference's environment), not in this package and not in its test suite -- like tools/load_into_sb3.py.  `--task` gives
the observation / action spaces of the stand-in env VecNormalize.load needs (hover 20 -> 4, yaw 12 -> 1); the env is never
stepped."""
import argparse

import numpy as np


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("pkl", help="VecNormalize pickle written by env.save / CheckpointCallback")
    ap.add_argument("out", help="the .npz to write")
    ap.add_argument("--task", choices=["hover", "yaw"], default="hover")
    args = ap.parse_args()

    import gymnasium as gym
    from stable_baselines3.common.vec_env import DummyVecEnv, VecNormalize

    obs_dim, act_dim = (20, 4) if args.task == "hover" else (12, 1)

    class Stand(gym.Env):
        observation_space = gym.spaces.Box(-np.inf, np.inf, (obs_dim,), np.float64)
        action_space = gym.spaces.Box(-1.0, 1.0, (act_dim,), np.float64)

        def reset(self, *, seed=None, options=None):
            return np.zeros(obs_dim), {}

        def step(self, action):
            return np.zeros(obs_dim), 0.0, False, False, {}

    vn = VecNormalize.load(args.pkl, DummyVecEnv([Stand]))
    flat = {}
    for name in ("obs_rms", "ret_rms"):
        rms = getattr(vn, name)
        flat[f"{name}.mean"], flat[f"{name}.var"], flat[f"{name}.count"] = np.asarray(rms.mean), np.asarray(rms.var), np.asarray(float(rms.count))
    for k in ("clip_obs", "clip_reward", "gamma", "epsilon", "norm_obs", "norm_reward"):
        flat[k] = np.asarray(getattr(vn, k))
    np.savez(args.out, **flat)
    print(f"{args.out}: obs_rms over {obs_dim} columns, count {float(vn.obs_rms.count):.0f}, clip_obs {vn.clip_obs}, norm_obs {vn.norm_obs}")


if __name__ == "__main__":
    main()
