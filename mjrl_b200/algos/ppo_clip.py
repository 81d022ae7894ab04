"""PPO with the clipped surrogate, with the reference's constructor and train_from_paths (mjrl/algos/ppo_clip.py:23-121).

`train_from_paths` whitens the advantages on the device, evaluates the surrogate, draws every minibatch index up front
(the reference's np.random.choice calls, value for value) and runs the whole epochs x N/mb_size chain of Adam steps as
ONE kernel launch (csrc/policy_sgd.cu); then surrogate and KL of the unclamped parameters, and the policy object takes
them (log_std clamped, as set_param_values does)."""
import time as timer

import numpy as np

from mjrl_b200.algos.batch_reinforce import BatchREINFORCE
from mjrl_b200.algos.policy_adam import PolicyAdam


def minibatch_indices(num_samples, mb_size, epochs):
    """The reference's epochs x int(N / mb_size) draws of np.random.choice(N, size=mb_size) (ppo_clip.py:88-90,
    behavior_cloning.py:121-123) as ONE np.random.randint call on the global RandomState: the legacy bounded-integer
    path consumes the generator per value and buffers nothing between calls, so the values and the generator state
    afterwards are the same.  Returns int32 [steps, mb_size]."""
    steps = epochs * int(num_samples / mb_size)
    idx = np.random.randint(0, num_samples, size=steps * mb_size)
    return idx.reshape(steps, mb_size).astype(np.int32)


def check_mlp_policy(policy, mb_size, who):
    if len(getattr(policy, "hidden_sizes", ())) != 2:
        raise NotImplementedError("%s runs on the Gaussian MLP policy (2 hidden layers); LinearPolicy is not supported" % who)
    if not 1 <= int(mb_size) <= 64:
        raise ValueError("%s: minibatch size must be in [1, 64] (the kernel holds one minibatch in shared memory)" % who)


class PPO(BatchREINFORCE):
    algo = "ppo"
    fit_overlap = False        # the reference draws the minibatch indices before the baseline fit's permutations

    def __init__(self, env, policy, baseline, clip_coef=0.2, epochs=10, mb_size=64, learn_rate=3e-4, seed=123,
                 save_logs=False, **kwargs):
        check_mlp_policy(policy, mb_size, "PPO")
        self._setup(env, policy, baseline, seed, save_logs)
        self.learn_rate, self.clip_coef, self.epochs, self.mb_size = learn_rate, clip_coef, epochs, mb_size
        self.adam = PolicyAdam(policy.d)              # torch.optim.Adam(policy.trainable_params, lr) (ppo_clip.py:46)
        self.record_minibatch_stats = False           # keep every step's minibatch loss / clip fraction (costs a little)
        self.last_minibatch_loss = self.last_clip_frac = None

    def update_from_rollouts(self, *args, **kwargs):
        raise NotImplementedError("PPO draws its minibatches before the baseline fit's permutations; the device-rollout "
                                  "path starts the fit first.  Use update_from_paths")

    def train_from_paths(self, paths):
        """ppo_clip.py:58-121."""
        _, _, _, base_stats, self.running_score = self.process_paths(paths)
        eng = self._engine
        if self.save_logs:
            self.log_rollout_statistics(paths, base_stats)
        surr_before = eng.eval()[0]
        ts = timer.time()
        idx = minibatch_indices(eng.n, self.mb_size, self.epochs)
        if len(idx):
            self.adam.bind(eng)
            out = eng.policy_sgd("ppo", idx, self.learn_rate, self.clip_coef, want_outputs=self.record_minibatch_stats)
            self.adam.pull(eng)
            if out is not None:
                self.last_minibatch_loss, self.last_clip_frac = out
        params_after = eng.get_params()
        surr_after, kl_dist = eng.eval()              # unclamped parameters, as the reference evaluates them
        self.policy.set_param_values(params_after, set_new=True, set_old=True)
        self._pushed = None
        t_opt = timer.time() - ts
        self.last_stats = dict(surr_before=surr_before, surr_after=surr_after, kl_dist=kl_dist)
        if self.save_logs:
            self.logger.log_kv('t_opt', t_opt)
            self.logger.log_kv('kl_dist', kl_dist)
            self.logger.log_kv('surr_improvement', surr_after - surr_before)
            self.logger.log_kv('running_score', self.running_score)
            if paths is not None:
                self._log_success(paths)
        return base_stats
