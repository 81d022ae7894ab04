"""TEST INFRASTRUCTURE: golden vectors of the reference's PPO-clip and behaviour cloning, produced by importing the
UNMODIFIED reference (oracle/ref_shim.py) on CPU:

    python -m oracle.make_golden_ppo_bc        ->  tests/golden/ppo_*.npz, tests/golden/bc_*.npz

Per case: theta_0 (after the agent's constructor), then after each of TWO consecutive calls (PPO: train_from_paths on two
batches; BC: train() twice) theta, the Adam moments / step count of the agent's optimizer, surr_before / surr_after /
kl_dist (PPO) or loss_before / loss_after (BC), and the per-step minibatch losses (PPO also the fraction of rows whose
gradient the clip zeroed).  Per-step values are recorded by subclasses that only observe.  Inputs are regenerated from
seeds (oracle.npg_oracle.synthetic_paths); arrays larger than FULL_MAX entries are stored as a seeded sample plus
per-parameter-block norms.  The files are written without timestamps, so a rerun reproduces them byte for byte."""
import io
import os
import sys
import zipfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from oracle import npg_oracle as O  # noqa: E402
from oracle import ppo_bc_oracle as PB  # noqa: E402
from oracle import ref_shim  # noqa: E402

GOLDEN_DIR = os.path.join(os.path.dirname(HERE), "tests", "golden")
FULL_MAX = 6000            # entries stored whole; larger vectors: SAMPLE entries + block norms
SAMPLE = 1024

CASES = {
    "ppo_17x6_h128": dict(kind="ppo", obs_dim=17, act_dim=6, hidden=(128, 128), n_paths=8, horizon=200, ragged=True,
                          epochs=2, mb=64, lr=3e-4, clip=0.2),
    "ppo_6x2_h32": dict(kind="ppo", obs_dim=6, act_dim=2, hidden=(32, 32), n_paths=4, horizon=120, ragged=False,
                        epochs=3, mb=64, lr=3e-4, clip=0.2),
    "ppo_clipheavy_6x2_h64": dict(kind="ppo", obs_dim=6, act_dim=2, hidden=(64, 64), n_paths=4, horizon=160, ragged=True,
                                  epochs=6, mb=48, lr=2e-2, clip=0.2),
    "ppo_39x28_h256": dict(kind="ppo", obs_dim=39, act_dim=28, hidden=(256, 256), n_paths=3, horizon=150, ragged=False,
                           epochs=1, mb=64, lr=3e-4, clip=0.2),
    "bc_mse_17x6_h128": dict(kind="bc", loss="MSE", obs_dim=17, act_dim=6, hidden=(128, 128), n_paths=6, horizon=200,
                             ragged=True, epochs=2, mb=64, lr=1e-3, set_transforms=False),
    "bc_mle_tr_11x3_h64": dict(kind="bc", loss="MLE", obs_dim=11, act_dim=3, hidden=(64, 64), n_paths=5, horizon=150,
                               ragged=True, epochs=3, mb=50, lr=1e-3, set_transforms=True),
}
POLICY_SEED, PATH_SEED, ADV_SEED, RNG_SEED = 500, 7, 11, 3


def store(out, key, a, cfg):
    """Whole, or (large) the entries at seeded positions + the norm of every parameter block."""
    a = np.ascontiguousarray(a, np.float32)
    if a.size <= FULL_MAX:
        out[key] = a
        return
    idx = np.sort(np.random.RandomState(0).choice(a.size, SAMPLE, replace=False))
    out[key + "@sample"] = a[idx]
    b = PB.block_bounds(cfg)
    out[key + "@norms"] = np.array([np.linalg.norm(a[lo:hi].astype(np.float64)) for lo, hi in zip(b[:-1], b[1:])])


def save_npz(path, arrays):
    """np.savez_compressed without the zip members' wall-clock timestamps (reproducible bytes)."""
    buf = io.BytesIO()
    with zipfile.ZipFile(buf, "w", compression=zipfile.ZIP_DEFLATED) as zf:
        for k in sorted(arrays):
            info = zipfile.ZipInfo(k + ".npy", date_time=(1980, 1, 1, 0, 0, 0))
            info.compress_type = zipfile.ZIP_DEFLATED
            with zf.open(info, "w") as f:
                np.lib.format.write_array(f, np.asanyarray(arrays[k]), allow_pickle=False)
    with open(path, "wb") as f:
        f.write(buf.getvalue())


def adam_flat(policy, opt):
    m, v, step = [], [], 0
    for p in policy.trainable_params:
        st = opt.state.get(p, {})
        m.append(st["exp_avg"].reshape(-1).numpy() if st else np.zeros(p.numel(), np.float32))
        v.append(st["exp_avg_sq"].reshape(-1).numpy() if st else np.zeros(p.numel(), np.float32))
        if st:
            step = max(step, int(st["step"]))
    return np.concatenate(m).astype(np.float32), np.concatenate(v).astype(np.float32), step


def run_ppo(R, PPO, cfg, meta):
    class RecPPO(PPO):
        """Observes the minibatch losses, clip fractions and the surrogate / KL values; changes nothing."""

        def PPO_surrogate(self, observations, actions, advantages):
            s = super().PPO_surrogate(observations, actions, advantages)
            with torch.no_grad():
                adv = torch.from_numpy(advantages).float()
                LR = self.policy.likelihood_ratio(self.policy.new_dist_info(observations, actions),
                                                  self.policy.old_dist_info(observations, actions))
                c = self.clip_coef
                live = ((LR >= 1 - c) & (LR <= 1 + c)) | (LR * adv < torch.clamp(LR, 1 - c, 1 + c) * adv)
                self.rec_clip.append(1.0 - float(live.float().mean()))
            self.rec_loss.append(-float(s.detach()))
            return s

        def CPI_surrogate(self, observations, actions, advantages):
            s = super().CPI_surrogate(observations, actions, advantages)
            self.rec_surr.append(float(s.detach()))
            return s

        def kl_old_new(self, observations, actions):
            k = super().kl_old_new(observations, actions)
            self.rec_kl.append(float(k.detach()))
            return k

    spec = R.EnvSpec(cfg["obs_dim"], cfg["act_dim"], cfg["horizon"])
    pol = R.MLP(spec, hidden_sizes=cfg["hidden"], seed=POLICY_SEED)
    agent = RecPPO(None, pol, None, clip_coef=cfg["clip"], epochs=cfg["epochs"], mb_size=cfg["mb"],
                   learn_rate=cfg["lr"], save_logs=False)
    out = {}
    store(out, "theta0", pol.get_param_values(), cfg)
    np.random.seed(RNG_SEED)
    for call in range(2):
        agent.rec_loss, agent.rec_clip, agent.rec_surr, agent.rec_kl = [], [], [], []
        paths = PB.case_paths(meta, call)
        agent.train_from_paths(paths)
        m, v, step = adam_flat(pol, agent.optimizer)
        store(out, "theta%d" % (call + 1), pol.get_param_values(), cfg)
        store(out, "m%d" % (call + 1), m, cfg)
        store(out, "v%d" % (call + 1), v, cfg)
        out["step%d" % (call + 1)] = np.int64(step)
        out["surr%d" % (call + 1)] = np.array(agent.rec_surr)          # before, after
        out["kl%d" % (call + 1)] = np.float64(agent.rec_kl[0])
        out["loss%d" % (call + 1)] = np.array(agent.rec_loss, np.float32)
        out["clipfrac%d" % (call + 1)] = np.array(agent.rec_clip, np.float32)
    out["rng_after"] = np.random.randint(0, 1 << 30, size=4)
    return out


def run_bc(R, BC, cfg, meta):
    class RecBC(BC):
        def loss(self, data, idx=None):
            val = super().loss(data, idx)
            if not isinstance(idx, range):
                self.rec_loss.append(float(val.detach()))
            return val

    spec = R.EnvSpec(cfg["obs_dim"], cfg["act_dim"], cfg["horizon"])
    pol = R.MLP(spec, hidden_sizes=cfg["hidden"], seed=POLICY_SEED)
    paths = PB.case_paths(meta, 0)
    agent = RecBC(paths, pol, epochs=cfg["epochs"], batch_size=cfg["mb"], lr=cfg["lr"], loss_type=cfg["loss"],
                  set_transforms=cfg["set_transforms"])
    out = {}
    store(out, "theta0", pol.get_param_values(), cfg)
    if cfg["set_transforms"]:
        for k in ("in_shift", "in_scale", "out_shift", "out_scale"):
            out[k] = getattr(pol.model, k).numpy().astype(np.float32)
    np.random.seed(RNG_SEED)
    for call in range(2):
        agent.rec_loss = []
        agent.train(suppress_fit_tqdm=True)
        m, v, step = adam_flat(pol, agent.optimizer)
        store(out, "theta%d" % (call + 1), pol.get_param_values(), cfg)
        store(out, "m%d" % (call + 1), m, cfg)
        store(out, "v%d" % (call + 1), v, cfg)
        out["step%d" % (call + 1)] = np.int64(step)
        out["bcloss%d" % (call + 1)] = np.array([agent.logger.log["loss_before"][-1], agent.logger.log["loss_after"][-1]])
        out["loss%d" % (call + 1)] = np.array(agent.rec_loss, np.float32)
    out["rng_after"] = np.random.randint(0, 1 << 30, size=4)
    return out


def main():
    R = ref_shim.load()
    from mjrl.algos.behavior_cloning import BC
    from mjrl.algos.ppo_clip import PPO
    torch.set_num_threads(1)
    for name, cfg in CASES.items():
        meta = dict(cfg, policy_seed=POLICY_SEED, path_seed=PATH_SEED, adv_seed=ADV_SEED, rng_seed=RNG_SEED)
        out = run_ppo(R, PPO, cfg, meta) if cfg["kind"] == "ppo" else run_bc(R, BC, cfg, meta)
        out["meta"] = np.array(repr(meta))
        path = os.path.join(GOLDEN_DIR, name + ".npz")
        save_npz(path, out)
        extra = ("  clipfrac %.2f" % float(np.mean(out["clipfrac1"]))) if cfg["kind"] == "ppo" else ""
        print("%-26s steps %d/%d%s  %.0f KB" % (name, len(out["loss1"]), len(out["loss2"]), extra,
                                               os.path.getsize(path) / 1024))


if __name__ == "__main__":
    main()
