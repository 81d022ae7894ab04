"""Behaviour cloning with the reference's constructor, fit and train (mjrl/algos/behavior_cloning.py:15-142).

The expert pairs go up as one flat batch; the epochs x N/batch_size chain of Adam steps on the MLE or MSE loss runs as
ONE kernel launch (csrc/policy_sgd.cu), and loss_before / loss_after are full-batch reductions on the device."""
import time as timer

import numpy as np

from mjrl_b200 import runtime
from mjrl_b200.algos.batch_reinforce import BatchREINFORCE
from mjrl_b200.algos.policy_adam import PolicyAdam
from mjrl_b200.algos.ppo_clip import check_mlp_policy, minibatch_indices
from mjrl_b200.utils.logger import DataLog

LOSSES = {'MLE': "mle", 'MSE': "mse"}


def _host(x):
    try:
        import torch
        if torch.is_tensor(x):
            return x.detach().cpu().numpy()
    except ImportError:      # pragma: no cover
        pass
    return np.asarray(x)


class BC:
    _push_policy = BatchREINFORCE._push_policy        # same device copy of (theta, transforms) as the RL agents

    def __init__(self, expert_paths, policy, epochs=5, batch_size=64, lr=1e-3, optimizer=None, loss_type='MSE',
                 save_logs=True, set_transforms=False, **kwargs):
        if optimizer is not None:
            raise NotImplementedError("BC runs torch.optim.Adam(policy.trainable_params, lr) on the GPU; a custom "
                                      "optimizer object cannot be executed there")
        if loss_type not in LOSSES:
            raise ValueError("loss_type must be 'MLE' or 'MSE', got %r" % (loss_type,))
        check_mlp_policy(policy, batch_size, "BC")
        self.policy, self.expert_paths = policy, expert_paths
        self.epochs, self.mb_size, self.lr = epochs, batch_size, lr
        self.logger = DataLog()
        self.loss_type, self.save_logs = loss_type, save_logs
        self.adam = PolicyAdam(policy.d)
        self.record_minibatch_stats = False           # keep every step's minibatch loss (costs a little)
        self.last_minibatch_loss = None
        self._engine, self._pushed = None, None
        if set_transforms:
            in_shift, in_scale, out_shift, out_scale = self.compute_transformations()
            self.set_transformations(in_shift, in_scale, out_shift, out_scale)
            self.set_variance_with_data(out_scale)

    # ---- reference helpers (behavior_cloning.py:52-72) ----
    def compute_transformations(self):
        if self.expert_paths == [] or self.expert_paths is None:
            return None, None, None, None
        observations = np.concatenate([path["observations"] for path in self.expert_paths])
        actions = np.concatenate([path["actions"] for path in self.expert_paths])
        return np.mean(observations, axis=0), np.std(observations, axis=0), np.mean(actions, axis=0), np.std(actions, axis=0)

    def set_transformations(self, in_shift=None, in_scale=None, out_shift=None, out_scale=None):
        self.policy.model.set_transformations(in_shift, in_scale, out_shift, out_scale)
        self.policy.old_model.set_transformations(in_shift, in_scale, out_shift, out_scale)
        self._pushed = None

    def set_variance_with_data(self, out_scale):
        params = self.policy.get_param_values()
        params[-self.policy.m:] = np.log(out_scale + 1e-12)
        self.policy.set_param_values(params)
        self._pushed = None

    # ---- engine ----
    def _eng(self, n):
        pol = self.policy
        eng = runtime.get_engine(pol.n, pol.m, pol.hidden_sizes, (128, 128), float(pol.min_log_std), need_samples=n,
                                 need_paths=1)
        if eng is not self._engine or getattr(eng, "policy_owner", None) is not self:
            self._engine, self._pushed = eng, None
            eng.policy_owner = self
        return eng

    def fit(self, data, suppress_fit_tqdm=False, **kwargs):
        """behavior_cloning.py:107-136 (data: dict of numpy arrays or CPU tensors, keys observations / expert_actions)."""
        assert all(k in data.keys() for k in ["observations", "expert_actions"])
        ts = timer.time()
        obs, act = _host(data["observations"]), _host(data["expert_actions"])
        n = obs.shape[0]
        eng = self._eng(n)
        eng.session_paths = None
        eng.upload_flat(obs, act, np.zeros(n), np.array([n], np.int32), np.zeros(1, np.uint8))
        self._push_policy(eng)
        kind = LOSSES[self.loss_type]
        if self.save_logs:
            self.logger.log_kv('loss_before', eng.bc_loss(kind))
        idx = minibatch_indices(n, self.mb_size, self.epochs)
        if len(idx):
            self.adam.bind(eng)
            out = eng.policy_sgd(kind, idx, self.lr, want_outputs=self.record_minibatch_stats)
            self.adam.pull(eng)
            if out is not None:
                self.last_minibatch_loss = out[0]
        self.policy.set_param_values(eng.get_params(), set_new=True, set_old=True)
        self._pushed = None
        if self.save_logs:
            self.logger.log_kv('epoch', self.epochs)
            self._push_policy(eng)                     # loss_after of the clamped parameters, as the reference
            self.logger.log_kv('loss_after', eng.bc_loss(kind))
            self.logger.log_kv('time', timer.time() - ts)

    def train(self, **kwargs):
        observations = np.concatenate([path["observations"] for path in self.expert_paths])
        expert_actions = np.concatenate([path["actions"] for path in self.expert_paths])
        self.fit(dict(observations=observations, expert_actions=expert_actions), **kwargs)
