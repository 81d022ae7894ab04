"""Host mirror of a policy optimizer's Adam state (torch.optim.Adam(policy.trainable_params) of PPO and BC).

The state belongs to the agent, as the reference's optimizer object does; the engine holds the working copy on the
device.  Engines are replaced when a larger batch arrives (runtime.get_engine) and agents may share one engine (BC
pre-training, then PPO or DAPG on the same policy), so the mirror is pulled after every chain and pushed again whenever
the engine changed or another agent's state was loaded into it since."""
import numpy as np


class PolicyAdam:
    def __init__(self, d):
        self.m, self.v, self.step = np.zeros(d, np.float32), np.zeros(d, np.float32), 0

    def bind(self, eng):
        if getattr(eng, "adam_owner", None) is not self:
            eng.adam_set(self.m, self.v, self.step)
            eng.adam_owner = self

    def pull(self, eng):
        self.m, self.v, self.step = eng.adam_get()

