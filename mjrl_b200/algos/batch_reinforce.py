"""Agent base class with the reference's orchestration (mjrl/algos/batch_reinforce.py:61-114, :178-214):
sample (host, mjrl's own samplers) -> returns -> advantages -> train_from_paths -> baseline.fit, with every
step after sampling executed by the CUDA engine."""
import time as timer

import numpy as np

from mjrl_b200 import runtime
from mjrl_b200.utils import process_samples
from mjrl_b200.utils.logger import DataLog


class BatchREINFORCE:
    """Only the plumbing shared by NPG / TRPO / DAPG is implemented; the reference's plain-REINFORCE update with a
    `desired_kl` line search (batch_reinforce.py:117-176) is a first-order method outside the NPG path."""

    algo = "npg"
    # Start the baseline fit before train_from_paths, on the engine's side stream.  Only valid when the reference draws
    # nothing from numpy's global RNG inside train_from_paths before the fit's permutations (PPO does: its minibatches).
    fit_overlap = True

    def _setup(self, env, policy, baseline, seed, save_logs):
        self.env, self.policy, self.baseline = env, policy, baseline
        self.seed, self.save_logs = seed, save_logs
        self.running_score = None
        if save_logs:
            self.logger = DataLog()
        self._engine = None
        self._pushed = None

    # ------------------------------------------------------------------ engine plumbing
    def _eng(self, need_samples=0, need_paths=0):
        pol = self.policy
        vf_hidden = getattr(self.baseline, "hidden_sizes", (128, 128)) if hasattr(self.baseline, "_eng") else (128, 128)
        eng = runtime.get_engine(pol.n, pol.m, pol.hidden_sizes, vf_hidden, float(pol.min_log_std),
                                 need_samples=need_samples, need_paths=need_paths)
        if eng is not self._engine or getattr(eng, "policy_owner", None) is not self:
            # a different engine, or another agent pushed ITS policy into this engine since: push again
            self._engine, self._pushed = eng, None
            eng.policy_owner = self
        if hasattr(self.baseline, "_bind"):
            self.baseline._bind(eng)
        return eng

    def _push_policy(self, eng):
        """Device copy of (theta_new, theta_old, transforms) <- the host policy object, when it changed."""
        pol = self.policy
        new = pol.get_param_values()
        old = np.concatenate([p.contiguous().view(-1).data.numpy() for p in pol.old_params])
        tr = [np.asarray(getattr(m, k).numpy(), np.float32) for m in (pol.model, pol.old_model)
              for k in ("in_shift", "in_scale", "out_shift", "out_scale")]
        sig = (new.tobytes(), old.tobytes(), b"".join(t.tobytes() for t in tr))
        if self._pushed == sig:
            return
        default = all(np.all(t == (0.0 if i % 2 == 0 else 1.0)) for i, t in enumerate(tr))
        if not default or getattr(eng, "_custom_transforms", False):
            eng.set_transforms(*tr[:4], old=False)
            eng.set_transforms(*tr[4:], old=True)
            eng._custom_transforms = True
        if np.array_equal(new, old):
            eng.set_params(new, True, True)
        else:
            eng.set_params(new, True, False)
            eng.set_params(old, False, True)
        self._pushed = sig

    def _resident(self, paths):
        """The engine holding `paths` as its rollout batch: inside runtime.session (update_from_paths) the pinned batch
        is reused, everywhere else the trajectories are uploaded again -- like the reference, a call always works on
        the arrays it is handed."""
        n = int(sum(len(p["rewards"]) for p in paths))
        eng = self._eng(n + self._demo_samples(), len(paths))
        runtime.ensure_resident(eng, paths)
        self._push_policy(eng)
        return eng

    def _demo_samples(self):
        return 0

    def _flat_batch(self, observations, actions, advantages=None, token=None):
        """For the reference-signature helpers that take concatenated arrays: upload them as the rollout batch.  Always
        uploads, except for the holder of `token` = (engine, generation) of an upload it made itself with exactly these
        array objects (build_Hvp_eval's closure: ten products over one batch) while no other upload happened since."""
        n = observations.shape[0]
        eng = self._eng(n, 1)
        reuse = (token is not None and token[0] is eng and token[1] == eng.generation
                 and token[2] is observations and token[3] is actions)
        if not reuse:
            eng.session_paths = None
            eng.upload_flat(observations, actions, np.zeros(n), np.array([n], np.int32), np.zeros(1, np.uint8))
        self._push_policy(eng)
        if advantages is not None:
            eng.set_white(np.asarray(advantages, np.float32))   # the reference passes whitened advantages here
        return eng

    # ------------------------------------------------------------------ reference-signature helpers
    def CPI_surrogate(self, observations, actions, advantages):
        """batch_reinforce.py:40-46 -> python float (the reference returns a 0-dim tensor)."""
        return self._flat_batch(observations, actions, advantages).eval()[0]

    def kl_old_new(self, observations, actions):
        """batch_reinforce.py:48-52."""
        eng = self._flat_batch(observations, actions, np.zeros(observations.shape[0]))
        return eng.eval()[1]

    def flat_vpg(self, observations, actions, advantages):
        """batch_reinforce.py:54-58 -> fp32 (d,)."""
        return self._flat_batch(observations, actions, advantages).vpg()

    # ------------------------------------------------------------------ train_step
    def train_step(self, N, env=None, sample_mode='trajectories', horizon=1e6, gamma=0.995, gae_lambda=0.97,
                   num_cpu='max', env_kwargs=None):
        """batch_reinforce.py:61-114.  Sampling stays on the host in mjrl's own sampler (MuJoCo, out of scope)."""
        try:
            import mjrl.samplers.core as trajectory_sampler
        except Exception as exc:   # pragma: no cover - needs mjrl + gym + mujoco on the host
            raise ImportError("train_step() samples with mjrl.samplers.core, which needs mjrl/gym/mujoco installed; "
                              "use update_from_paths(paths) when you bring your own trajectories") from exc
        env = self.env.env_id if env is None else env
        if sample_mode not in ('trajectories', 'samples'):
            raise ValueError("sample_mode must be 'trajectories' or 'samples'")
        ts = timer.time()
        kw = dict(env=env, policy=self.policy, horizon=horizon, base_seed=self.seed, num_cpu=num_cpu, env_kwargs=env_kwargs)
        if sample_mode == 'trajectories':
            paths = trajectory_sampler.sample_paths(num_traj=N, **kw)
        else:
            paths = trajectory_sampler.sample_data_batch(num_samples=N, **kw)
        if self.save_logs:
            self.logger.log_kv('time_sampling', timer.time() - ts)
        self.seed = self.seed + N if self.seed is not None else self.seed
        stats = self.update_from_paths(paths, gamma, gae_lambda)
        stats.append(N)
        return stats

    def update_from_paths(self, paths, gamma=0.995, gae_lambda=0.97):
        """Everything train_step does after sampling (batch_reinforce.py:94-112) on one resident device batch."""
        n = int(sum(len(p["rewards"]) for p in paths))
        eng = self._eng(n + self._demo_samples(), len(paths))
        with runtime.session(eng, paths):                    # ONE upload per call, always; pinned for the nested helpers
            self._push_policy(eng)
            return self._update_resident(eng, paths, gamma, gae_lambda)

    def _update_resident(self, eng, paths, gamma, gae_lambda):
        # The sequential baseline fit is the longest chain of the step and depends only on the returns: it is started
        # right away on the engine's side stream; the write-back of the returns, the advantages (with the PRE-fit
        # baseline, as in the reference's program order) and the policy update run concurrently.  With
        # hvp_sample_frac < 1 the reference interleaves host RNG draws (one index set per Fisher product actually
        # evaluated, then the fit permutations, A9); that order is only reproducible with the fit AFTER the policy
        # step, so the overlap is switched off for that setting.
        subsampling = getattr(self, "hvp_subsample", None) is not None and self.hvp_subsample < 0.99
        overlap = self.fit_overlap and hasattr(self.baseline, "fit_begin") and not subsampling
        process_samples.returns_on(eng, paths, gamma, write_back=not overlap)
        error_before = error_after = None
        fit_started = False
        try:
            if overlap:
                self.baseline._bind(eng)
                error_before = self.baseline.fit_begin(paths, return_errors=self.save_logs)
                fit_started = True
                process_samples.returns_write_back(eng, paths)
            process_samples.advantages_on(eng, paths, self.baseline, gamma, gae_lambda, fit_in_flight=overlap)
            eval_statistics = self.train_from_paths(paths)
        except BaseException:
            if fit_started:                               # never leave a fit in flight behind a failed policy step
                try:
                    self.baseline.fit_end(return_errors=False)
                except Exception:
                    pass
            raise
        if self.save_logs:
            self.logger.log_kv('num_samples', int(np.sum([p["rewards"].shape[0] for p in paths])))
        ts = timer.time()
        if overlap and not self.save_logs and hasattr(self.baseline, "fit_defer"):
            # theta is back on the host: return now.  The fit keeps running on its own stream and is joined by whoever
            # reads the baseline next (predict / fit / pickling), so the next batch's upload overlaps its tail.
            self.baseline.fit_defer()
        elif overlap:
            error_after = self.baseline.fit_end(return_errors=self.save_logs)
        elif hasattr(self.baseline, "fit_resident"):      # ridge baselines: Gram pass over the resident batch + host solve
            errs = self.baseline.fit_resident(eng, return_errors=self.save_logs)
            if self.save_logs:
                error_before, error_after = errs
        elif self.save_logs:
            error_before, error_after = self.baseline.fit(paths, return_errors=True)
        else:
            self.baseline.fit(paths)
        if self.save_logs:
            # overlap mode: the fit ran concurrently with the policy update; time_VF is the wall time still spent
            # waiting for it after train_from_paths returned (the reference logs the whole sequential fit here)
            self.logger.log_kv('time_VF', timer.time() - ts)
            self.logger.log_kv('VF_error_before', error_before)
            self.logger.log_kv('VF_error_after', error_after)
        return eval_statistics

    def update_from_rollouts(self, rollouts, gamma=0.995, gae_lambda=0.97, lengths=None, terminated=None):
        """The post-rollout update on DEVICE-RESIDENT batched rollouts -- the hand-off the model-based caller wants
        (algos/model_accel/model_accel_npg.py:107-181: learned-model rollouts are already batched tensors
        `rollouts['observations'|'actions'|'rewards']` of shape [n_traj, horizon, ...], model_accel/sampling.py:16-90;
        the reference slices them into host path dicts and concatenates them again).  Here they are packed on the device
        (`mjb_batch_upload_rollouts`) and the whole step -- returns, GAE, whitening, VPG, CG, step, baseline fit -- runs
        without the samples ever visiting the host.  `lengths[i] <= horizon` keeps a prefix of trajectory i (termination
        function / ensemble truncation, :129-158), `terminated[i]` marks it as terminated for the GAE bootstrap.
        numpy arrays / CPU tensors are accepted and moved with torch.  Returns the reference's base_stats list."""
        import torch
        if not hasattr(self.baseline, "fit_begin_resident"):
            raise NotImplementedError("update_from_rollouts needs the device MLPBaseline (host baselines want path dicts)")
        if getattr(self, "input_normalization", None):
            raise NotImplementedError("input_normalization reads host observations: use update_from_paths")
        dev = torch.device("cuda", runtime.device_ordinal())
        tens = []
        for k in ("observations", "actions", "rewards"):
            x = rollouts[k]
            x = x if torch.is_tensor(x) else torch.as_tensor(np.asarray(x))
            tens.append(x.to(dev) if not x.is_cuda else x)
        dt = torch.float64 if any(t.dtype == torch.float64 for t in tens) else torch.float32
        obs, act, rew = (t.to(dt) for t in tens)
        n_traj, H = int(obs.shape[0]), int(obs.shape[1])
        n = int(np.sum(lengths)) if lengths is not None else n_traj * H
        eng = self._eng(n + self._demo_samples(), n_traj)
        eng.session_paths = None
        eng.upload_rollouts(obs, act, rew, lengths, terminated)
        self._push_policy(eng)
        eng.compute_returns(gamma)
        error_before = self.baseline.fit_begin_resident(eng, return_errors=self.save_logs)
        fit_started = True
        try:
            eng.vf_predict(prefit=True)                      # pre-fit baseline, as in the reference's program order
            eng.compute_advantages(gamma, gae_lambda)
            stats = self._train_resident(eng, None)
        except BaseException:
            if fit_started:
                try:
                    self.baseline.fit_end(return_errors=False)
                except Exception:
                    pass
            raise
        if self.save_logs:
            self.logger.log_kv('num_samples', n)
            ts = timer.time()
            error_after = self.baseline.fit_end(return_errors=True)
            self.logger.log_kv('time_VF', timer.time() - ts)
            self.logger.log_kv('VF_error_before', error_before)
            self.logger.log_kv('VF_error_after', error_after)
        else:
            self.baseline.fit_defer()
        return stats

    # ------------------------------------------------------------------ shared pieces of train_from_paths
    def process_paths(self, paths):
        """batch_reinforce.py:178-197: whitening + return statistics on the device; returns the reference's tuple
        except that the concatenated arrays stay on the GPU (None placeholders).  paths=None: the engine's resident
        batch with device-computed advantages (update_from_rollouts)."""
        if paths is None:
            eng = self._engine
            assert eng is not None and eng.adv_on_device
        else:
            eng = self._resident(paths)
            if "advantages" in paths[0] and not eng.adv_on_device:
                # anything but advantages the engine itself just computed for this very upload comes from the path dicts
                eng.set_advantages(np.concatenate([p["advantages"] for p in paths]))
        st = eng.process_paths()
        base_stats = [st.mean_return, st.std_return, st.min_return, st.max_return]
        running = st.mean_return if self.running_score is None else 0.9 * self.running_score + 0.1 * st.mean_return
        return None, None, None, base_stats, running

    def log_rollout_statistics(self, paths, base_stats=None):
        if base_stats is None:
            rets = [float(np.sum(p["rewards"])) for p in paths]
            base_stats = [np.mean(rets), np.std(rets), np.amin(rets), np.amax(rets)]
        self.logger.log_kv('stoc_pol_mean', base_stats[0])
        self.logger.log_kv('stoc_pol_std', base_stats[1])
        self.logger.log_kv('stoc_pol_max', base_stats[3])
        self.logger.log_kv('stoc_pol_min', base_stats[2])
        try:
            self.logger.log_kv('rollout_success', self.env.env.env.evaluate_success(paths))
        except Exception:
            pass

    def _log_success(self, paths):
        try:
            self.env.env.env.evaluate_success(paths, self.logger)
        except Exception:
            try:
                self.logger.log_kv('success_rate', self.env.env.env.evaluate_success(paths))
            except Exception:
                pass

    def _finish_step(self, eng, st, paths, t_host):
        """Pull theta back into the picklable host policy (new and old) and emit the reference's log keys."""
        new = eng.get_params()
        self.policy.set_param_values(new, set_new=True, set_old=True)
        self._pushed = None
        self.last_step = st
        if self.save_logs:
            self.logger.log_kv('alpha', st.alpha)
            self.logger.log_kv('delta', st.delta)
            self.logger.log_kv('time_vpg', st.time_vpg_ms * 1e-3)
            self.logger.log_kv('time_npg', st.time_npg_ms * 1e-3)
            self.logger.log_kv('kl_dist', st.kl_dist)
            self.logger.log_kv('surr_improvement', st.surr_after - st.surr_before)
            self.logger.log_kv('running_score', self.running_score)
            if paths is not None:
                self._log_success(paths)
