"""Timing of the minibatch-Adam policy chain (csrc/policy_sgd.cu) behind PPO and BC.

    python tools/ppo_bc_bench.py [--out FILE]

Prints one JSON line: microseconds per Adam step from CUDA events around the chain at the cfg2 / cfg3 / cfg4 policy
shapes, one full PPO.train_from_paths at cfg3 (1e6 samples, the reference's defaults: 10 epochs, minibatch 64), one
BC.fit at a DAPG demonstration size, and the card's name and power limit read in the same run.  Inputs are seeded."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = {"cfg2": (8, 2, (64, 64)), "cfg3": (17, 6, (128, 128)), "cfg4": (39, 28, (256, 256))}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, plim = [s.strip() for s in out.split(",")]
        return name, plim
    except Exception as exc:       # the numbers are still printed, marked as lacking the card's description
        return "unknown (%s)" % exc, "unknown"


def per_step_us(obs_dim, act_dim, hidden, n=200_000, steps=6000):
    from mjrl_b200.engine import Engine
    rng = np.random.RandomState(0)
    eng = Engine(obs_dim, act_dim, hidden, max_samples=n + 64, max_paths=8)
    eng.upload_flat(rng.randn(n, obs_dim), 0.1 * rng.randn(n, act_dim), np.zeros(n), np.array([n], np.int32),
                    np.zeros(1, np.uint8))
    eng.set_advantages(rng.randn(n))
    eng.process_paths()
    idx = rng.randint(0, n, size=(steps, 64)).astype(np.int32)
    out = {}
    for loss in ("ppo", "mse"):
        eng.policy_sgd(loss, idx[:200], 3e-4)                          # warm-up (module load, attribute set-up)
        eng.policy_sgd(loss, idx, 3e-4)
        out[loss] = round(1e3 * eng.last_sgd_ms() / steps, 3)
    eng.close()
    return out


def ppo_cfg3():
    from mjrl_b200 import runtime
    from mjrl_b200.algos.ppo_clip import PPO
    from mjrl_b200.policies.gaussian_mlp import MLP
    from mjrl_b200.utils.gym_env import EnvSpec
    rng = np.random.RandomState(1)
    paths = [dict(observations=rng.randn(1000, 17), actions=rng.randn(1000, 6), rewards=rng.randn(1000),
                  advantages=rng.randn(1000)) for _ in range(1000)]
    pol = MLP(EnvSpec(17, 6, 1000), hidden_sizes=(128, 128), seed=0)
    agent = PPO(None, pol, None, save_logs=True)
    np.random.seed(0)
    agent.train_from_paths(paths[:16])                                 # warm-up on a small batch (same engine shape)
    t0 = time.time()
    agent.train_from_paths(paths)
    wall = time.time() - t0
    eng = agent._engine
    steps = 10 * (1_000_000 // 64)
    res = dict(samples=1_000_000, adam_steps=steps, train_from_paths_s=round(wall, 3),
               chain_ms=round(eng.last_sgd_ms(), 1), us_per_step=round(1e3 * eng.last_sgd_ms() / steps, 3),
               t_opt_s=round(agent.logger.log["t_opt"][-1], 3), kl_dist=agent.logger.log["kl_dist"][-1],
               surr_improvement=agent.logger.log["surr_improvement"][-1])
    runtime.shutdown()
    return res


def bc_demo():
    from mjrl_b200 import runtime
    from mjrl_b200.algos.behavior_cloning import BC
    from mjrl_b200.policies.gaussian_mlp import MLP
    from mjrl_b200.utils.gym_env import EnvSpec
    rng = np.random.RandomState(2)
    demos = [dict(observations=rng.randn(200, 39), actions=rng.randn(200, 28)) for _ in range(25)]
    pol = MLP(EnvSpec(39, 28, 200), hidden_sizes=(32, 32), seed=0)
    bc = BC(demos, pol, epochs=5, batch_size=64, lr=1e-3, loss_type='MSE', set_transforms=False)
    np.random.seed(0)
    bc.train()                                                         # warm-up
    bc.train()
    res = dict(demo_rows=5000, obs_dim=39, act_dim=28, hidden=[32, 32], epochs=5, adam_steps=5 * (5000 // 64),
               fit_s=round(bc.logger.log["time"][-1], 4), chain_ms=round(bc._engine.last_sgd_ms(), 2),
               loss_before=bc.logger.log["loss_before"][-1], loss_after=bc.logger.log["loss_after"][-1])
    runtime.shutdown()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    name, plim = card()
    res = dict(card=name, power_limit=plim,
               us_per_adam_step={k: per_step_us(*v) for k, v in SHAPES.items()},
               ppo_cfg3_train_from_paths=ppo_cfg3(), bc_fit_dapg_demo=bc_demo())
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
