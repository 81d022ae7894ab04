"""Python handle over the C-ABI engine (include/mjrl_b200.h).  Host arrays are numpy; device memory,
streams and kernels live behind the library.  torch is used only for torch.distributed plumbing
(broadcasting the NCCL unique id when world_size > 1)."""
import ctypes as C

import numpy as np

from . import _native
from ._native import BatchStats, Config, MjbError, StepStats

ALGO = {"npg": 0, "trpo": 1, "dapg": 2}
LOSS = {"ppo": 0, "mle": 1, "mse": 2}
ROLLOUT, DEMO = 0, 1


def _ptr(a):
    return C.c_void_p(a.ctypes.data) if a is not None else None


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


class Engine:
    """One engine per GPU / per rank.  Not thread-safe (neither is mjrl)."""

    def __init__(self, obs_dim, act_dim, hidden=(64, 64), vf_hidden=(128, 128), min_log_std=-3.0,
                 max_samples=1 << 16, max_paths=4096, device=0, world_size=1, rank=0):
        self.lib = _native.load()
        self.p2p = False          # fused peer-memory all-reduce of the Fisher products (set by init_p2p, world_size > 1)
        hidden = tuple(int(h) for h in hidden)
        if len(hidden) not in (0, 2):
            raise NotImplementedError("mjrl_b200 supports LinearPolicy (no hidden layer) and 2-hidden-layer MLPs "
                                      "(the reference MLP is '2 layers only', gaussian_mlp.py:15)")
        cfg = Config()
        cfg.device, cfg.obs_dim, cfg.act_dim, cfg.n_hidden = int(device), int(obs_dim), int(act_dim), len(hidden)
        for i, h in enumerate(hidden):
            cfg.hidden[i] = h
        cfg.vf_hidden[0], cfg.vf_hidden[1] = int(vf_hidden[0]), int(vf_hidden[1])
        cfg.min_log_std = float(min_log_std)
        cfg.max_samples, cfg.max_paths = int(max_samples), int(max_paths)
        cfg.world_size, cfg.rank = int(world_size), int(rank)
        self.cfg = cfg
        self.obs_dim, self.act_dim, self.hidden, self.vf_hidden = int(obs_dim), int(act_dim), hidden, tuple(vf_hidden)
        self.max_samples, self.max_paths = int(max_samples), int(max_paths)
        self.world_size, self.rank = int(world_size), int(rank)
        h = C.c_void_p()
        if self.lib.mjb_create(C.byref(cfg), C.byref(h)) != 0:
            raise MjbError("mjb_create: " + self.lib.mjb_last_error(None).decode())
        self._h = h
        self.d = self.lib.mjb_policy_dim(h)
        self.vf_d = self.lib.mjb_vf_dim(h)
        self.n = 0
        self.n_demo = 0
        # residency bookkeeping of the Python mirror (runtime.session / BatchREINFORCE._flat_batch)
        self.generation = 0            # bumped by every rollout upload
        self.session_paths = None      # the list object pinned by runtime.session (strong reference, compared with `is`)
        self.have_returns = False      # device returns valid for the resident batch
        self.adv_on_device = False     # device advantages were computed by the engine for the resident batch

    # ------------------------------------------------------------------ plumbing
    @property
    def h(self):
        """The C handle; a closed engine fails loudly instead of passing NULL into the C ABI."""
        if self._h is None:
            raise MjbError("this Engine was closed (runtime.get_engine replaced it with a larger one); "
                           "re-resolve it through runtime.get_engine")
        return self._h

    @property
    def closed(self):
        return self._h is None

    def close(self):
        if getattr(self, "_h", None):
            self.lib.mjb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc, what):
        if rc != 0:
            raise MjbError("%s: %s" % (what, self.lib.mjb_last_error(self.h).decode()))

    def synchronize(self):
        self._ck(self.lib.mjb_synchronize(self.h), "synchronize")

    def init_comm(self):
        """Create the engine-owned NCCL communicator; the unique id travels over torch.distributed."""
        if self.world_size == 1:
            return
        from .parallel import broadcast_bytes
        buf = (C.c_char * 128)()
        if self.rank == 0 and self.lib.mjb_comm_unique_id(buf) != 0:
            raise MjbError("mjb_comm_unique_id: " + self.lib.mjb_last_error(None).decode())
        raw = broadcast_bytes(bytes(buf), 128, src=0, device=self.cfg.device)
        self._ck(self.lib.mjb_comm_init(self.h, C.c_char_p(raw)), "comm_init")
        self.init_p2p()

    def init_p2p(self):
        """All-reduce of the Fisher-vector products over NVLink peer memory (csrc/p2p.cu): the ranks exchange the CUDA IPC
        handles of their exchange buffers; the fused kernel is switched on only if EVERY rank could map every peer
        (otherwise all ranks stay on ncclAllReduce).  MJRL_B200_P2P=0 keeps NCCL."""
        import os
        from .parallel import all_gather_bytes, all_ranks_agree
        self.p2p = False
        want = os.environ.get("MJRL_B200_P2P", "1") != "0"
        h = (C.c_char * 64)()
        ok = want and self.lib.mjb_p2p_export(self.h, h) == 0
        handles = all_gather_bytes(bytes(h), 64, device=self.cfg.device)
        if ok:
            ok = self.lib.mjb_p2p_import(self.h, C.c_char_p(b"".join(handles))) == 0
        if all_ranks_agree(ok, device=self.cfg.device):
            self.p2p = bool(self.lib.mjb_p2p_enable(self.h, 1))

    def set_p2p(self, on):
        """Switch between the fused peer-memory all-reduce and ncclAllReduce (collective: call on every rank)."""
        self.p2p = bool(self.lib.mjb_p2p_enable(self.h, 1 if on else 0))
        return self.p2p

    def p2p_calls(self):
        return int(self.lib.mjb_p2p_calls(self.h))

    # ------------------------------------------------------------------ trajectories
    def upload_paths(self, paths, which=ROLLOUT):
        """paths: list of mjrl path dicts (samplers/core.py:85-92).  float64 arrays are passed by pointer."""
        n_paths = len(paths)
        keep, ptrs = [], []
        for key in ("observations", "actions", "rewards"):
            if key == "rewards" and which == DEMO:
                ptrs.append(None)
                continue
            arrs = [np.ascontiguousarray(p[key], dtype=np.float64) for p in paths]
            keep.append(arrs)
            ptrs.append((C.c_void_p * n_paths)(*[a.ctypes.data for a in arrs]))
        lens = np.array([len(p["actions"]) for p in paths], dtype=np.int32)
        term = np.array([bool(p.get("terminated", False)) for p in paths], dtype=np.uint8)
        self._ck(self.lib.mjb_batch_upload(self.h, which, n_paths, ptrs[0], ptrs[1], ptrs[2], _ptr(lens), _ptr(term)),
                 "batch_upload")
        self._uploaded(which, lens)
        return self.n

    def _uploaded(self, which, lens):
        if which == ROLLOUT:
            self.n, self.n_demo, self.lens = int(lens.sum()), 0, lens
            self.generation += 1
            self.have_returns = False
            self.adv_on_device = False
        else:
            self.n_demo = int(lens.sum())

    def upload_flat(self, obs, act, rew, lens, terminated, which=ROLLOUT):
        obs = np.ascontiguousarray(obs, dtype=np.float64)
        act = np.ascontiguousarray(act, dtype=np.float64)
        rew = None if rew is None else np.ascontiguousarray(rew, dtype=np.float64)
        lens = np.ascontiguousarray(lens, dtype=np.int32)
        term = np.ascontiguousarray(terminated, dtype=np.uint8)
        self._ck(self.lib.mjb_batch_upload_flat(self.h, which, len(lens), _ptr(obs), _ptr(act), _ptr(rew), _ptr(lens),
                                                _ptr(term)), "batch_upload_flat")
        self._uploaded(which, lens)
        return self.n

    def upload_rollouts(self, obs, act, rew, lens=None, terminated=None):
        """Device-resident batched rollouts: torch CUDA tensors obs [n, H, obs_dim], act [n, H, act_dim], rew [n, H]
        (float32 or float64, all the same dtype).  lens (optional, <= H per trajectory) keeps prefixes."""
        import torch
        assert obs.is_cuda and act.is_cuda and rew.is_cuda, "upload_rollouts takes CUDA tensors"
        assert obs.dtype == act.dtype == rew.dtype and obs.dtype in (torch.float32, torch.float64)
        obs, act, rew = obs.contiguous(), act.contiguous(), rew.contiguous()
        n_traj, H = int(obs.shape[0]), int(obs.shape[1])
        assert obs.shape[2] == self.obs_dim and act.shape[2] == self.act_dim and tuple(rew.shape) == (n_traj, H)
        lens_a = np.full(n_traj, H, np.int32) if lens is None else np.ascontiguousarray(lens, dtype=np.int32)
        term = np.zeros(n_traj, np.uint8) if terminated is None else np.ascontiguousarray(terminated, dtype=np.uint8)
        torch.cuda.current_stream(obs.device).synchronize()       # the producers of the tensors are done
        self._ck(self.lib.mjb_batch_upload_rollouts(self.h, n_traj, H, C.c_void_p(obs.data_ptr()), C.c_void_p(act.data_ptr()),
                                                    C.c_void_p(rew.data_ptr()), int(obs.dtype == torch.float64), _ptr(lens_a),
                                                    _ptr(term)), "batch_upload_rollouts")
        self.synchronize()                                        # the tensors may be freed / reused by the caller now
        self._uploaded(ROLLOUT, lens_a)
        return self.n

    def set_advantages(self, adv_concat):
        a = np.ascontiguousarray(adv_concat, dtype=np.float64)
        assert a.shape[0] == self.n
        self._ck(self.lib.mjb_batch_set_advantages(self.h, _ptr(a)), "set_advantages")
        self.adv_on_device = False

    def set_white(self, adv_white):
        w = _f32(adv_white)
        assert w.shape[0] == self.n
        self._ck(self.lib.mjb_batch_set_adv_white(self.h, _ptr(w)), "set_adv_white")

    def set_returns(self, ret_concat):
        r = np.ascontiguousarray(ret_concat, dtype=np.float64)
        assert r.shape[0] == self.n
        self._ck(self.lib.mjb_batch_set_returns(self.h, _ptr(r)), "set_returns")
        self.have_returns = True

    def n_global(self):
        return int(self.lib.mjb_batch_size(self.h, 2))

    def set_baseline(self, base_concat):
        b = _f32(base_concat)
        assert b.shape[0] == self.n
        self._ck(self.lib.mjb_batch_set_baseline(self.h, _ptr(b)), "set_baseline")

    # ------------------------------------------------------------------ returns / advantages
    def compute_returns(self, gamma):
        self._ck(self.lib.mjb_compute_returns(self.h, float(gamma)), "compute_returns")
        self.have_returns = True

    def vf_predict(self, prefit=False):
        """prefit=True: predictions with the baseline of the last completed fit, without joining a fit in flight."""
        if prefit:
            self._ck(self.lib.mjb_vf_predict_prefit(self.h), "vf_predict_prefit")
        else:
            self._ck(self.lib.mjb_vf_predict(self.h), "vf_predict")

    # ------------------------------------------------------------------ ridge baselines (csrc/ridge.cu)
    def ridge_features(self, kind):
        return int(self.lib.mjb_ridge_features(self.h, int(kind)))

    def ridge_gram(self, kind):
        """Gram matrix of [features | returns] over the resident batch (all ranks): (F^T F [K,K], F^T y [K], y^T y)."""
        K = self.ridge_features(kind)
        out = np.empty((K + 1, K + 1), dtype=np.float64)
        self._ck(self.lib.mjb_ridge_gram(self.h, int(kind), out.ctypes.data_as(C.c_void_p)), "ridge_gram")
        return out[:K, :K].copy(), out[:K, K].copy(), float(out[K, K])

    def ridge_predict(self, kind, coeffs, want_sq_err=False):
        """features . coeffs for every resident sample into the device baseline buffer; optionally sum (returns - pred)^2."""
        c = np.ascontiguousarray(coeffs, dtype=np.float64)
        if c.shape != (self.ridge_features(kind),):
            raise ValueError("ridge_predict: %d coefficients expected" % self.ridge_features(kind))
        err = C.c_double(0.0)
        self._ck(self.lib.mjb_ridge_predict(self.h, int(kind), c.ctypes.data_as(C.c_void_p),
                                            C.byref(err) if want_sq_err else None), "ridge_predict")
        return float(err.value) if want_sq_err else None

    def compute_advantages(self, gamma, gae_lambda):
        use_gae = gae_lambda is not None and 0.0 <= gae_lambda <= 1.0
        self._ck(self.lib.mjb_compute_advantages(self.h, float(gamma), float(gae_lambda) if use_gae else 0.0,
                                                 int(use_gae)), "compute_advantages")
        self.adv_on_device = True

    def _get(self, fn, dtype):
        out = np.empty(self.n, dtype=dtype)
        self._ck(fn(self.h, _ptr(out)), fn.__name__)
        return out

    def returns(self):
        return self._get(self.lib.mjb_get_returns, np.float64)

    def baseline(self):
        return self._get(self.lib.mjb_get_baseline, np.float32)

    def advantages(self):
        return self._get(self.lib.mjb_get_advantages, np.float64)

    def adv_white(self):
        return self._get(self.lib.mjb_get_adv_white, np.float32)

    def process_paths(self):
        st = BatchStats()
        self._ck(self.lib.mjb_process_paths(self.h, C.byref(st)), "process_paths")
        return st

    # ------------------------------------------------------------------ policy
    def set_params(self, theta, set_new=True, set_old=True):
        th = _f32(theta)
        assert th.shape[0] == self.d, "parameter vector has %d entries, engine expects %d" % (th.shape[0], self.d)
        self._ck(self.lib.mjb_policy_set_params(self.h, _ptr(th), int(set_new), int(set_old)), "set_params")
        self.synchronize()

    def get_params(self, old=False):
        out = np.empty(self.d, dtype=np.float32)
        self._ck(self.lib.mjb_policy_get_params(self.h, _ptr(out), int(old)), "get_params")
        return out

    def set_transforms(self, in_shift=None, in_scale=None, out_shift=None, out_scale=None, old=False):
        arrs = [None if a is None else _f32(a) for a in (in_shift, in_scale, out_shift, out_scale)]
        self._ck(self.lib.mjb_policy_set_transforms(self.h, *[_ptr(a) for a in arrs], int(old)), "set_transforms")

    def eval(self):
        out = (C.c_double * 2)()
        self._ck(self.lib.mjb_policy_eval(self.h, C.byref(out)), "policy_eval")
        return out[0], out[1]

    def vpg(self, include_demo=False, demo_lam=0.0):
        g = np.empty(self.d, dtype=np.float32)
        self._ck(self.lib.mjb_policy_vpg(self.h, int(include_demo), float(demo_lam), _ptr(g)), "policy_vpg")
        return g

    def fvp(self, v, damping, idx=None):
        v = _f32(v)
        out = np.empty(self.d, dtype=np.float32)
        ii = None if idx is None else np.ascontiguousarray(idx, dtype=np.int32)
        self._ck(self.lib.mjb_policy_fvp(self.h, _ptr(v), float(damping), _ptr(ii), 0 if ii is None else ii.shape[0],
                                         _ptr(out)), "policy_fvp")
        return out

    def cg(self, b=None, iters=10, damping=1e-4, tol=1e-10, idx=None):
        bb = None if b is None else _f32(b)
        x = np.empty(self.d, dtype=np.float32)
        ii = None if idx is None else np.ascontiguousarray(idx, dtype=np.int32).reshape(iters, -1)
        self._ck(self.lib.mjb_policy_cg(self.h, _ptr(bb), int(iters), float(damping), float(tol), _ptr(ii),
                                        0 if ii is None else ii.shape[1], _ptr(x)), "policy_cg")
        return x

    def step(self, algo="npg", step_size=0.01, const_learn_rate=None, cg_iters=10, damping=1e-4, demo_lam=0.0,
             hvp_idx=None):
        st = StepStats()
        if isinstance(hvp_idx, (list, tuple)):               # ragged per-iteration lists (data-parallel subsample)
            lens = np.array([len(r) for r in hvp_idx], dtype=np.int64)
            stride = max(1, int(lens.max()))
            block = np.zeros((cg_iters, stride), dtype=np.int32)
            for i, r in enumerate(hvp_idx):
                block[i, :len(r)] = r
            self._ck(self.lib.mjb_policy_set_hvp_lengths(self.h, _ptr(lens), int(cg_iters)), "set_hvp_lengths")
            hvp_idx = block
        ii = None if hvp_idx is None else np.ascontiguousarray(hvp_idx, dtype=np.int32).reshape(cg_iters, -1)
        self._ck(self.lib.mjb_policy_step(self.h, ALGO[algo], float(step_size),
                                          -1.0 if const_learn_rate is None else float(const_learn_rate),
                                          int(cg_iters), float(damping), float(demo_lam), _ptr(ii),
                                          0 if ii is None else ii.shape[1], C.byref(st)), "policy_step")
        return st

    # ------------------------------------------------------------------ minibatch-Adam policy training (PPO, BC)
    def policy_sgd(self, loss, idx, lr, clip_coef=0.2, want_outputs=False):
        """Sequential Adam steps on theta_new (csrc/policy_sgd.cu), one minibatch per row of idx [steps, batch] (rows of
        the resident batch).  loss: "ppo", "mle" or "mse".  want_outputs: also return every step's minibatch loss and
        (PPO) the fraction of the minibatch the clip zeroed, as two float32 arrays."""
        ii = np.ascontiguousarray(idx, dtype=np.int32)
        if ii.ndim != 2:
            raise ValueError("policy_sgd: idx must be [steps, batch]")
        steps, batch = ii.shape
        if ii.size and (int(ii.min()) < 0 or int(ii.max()) >= self.n):
            raise ValueError("policy_sgd: minibatch index outside the resident batch of %d rows" % self.n)
        loss_out = np.empty(steps, np.float32) if want_outputs else None
        clip_out = np.empty(steps, np.float32) if want_outputs else None
        self._ck(self.lib.mjb_policy_sgd(self.h, LOSS[loss], _ptr(ii), int(steps), int(batch), float(lr), float(clip_coef),
                                         _ptr(loss_out), _ptr(clip_out)), "policy_sgd")
        return (loss_out, clip_out) if want_outputs else None

    def adam_set(self, m=None, v=None, step=-1):
        arrs = [None if a is None else _f32(a) for a in (m, v)]
        for a in arrs:
            assert a is None or a.shape[0] == self.d
        self._ck(self.lib.mjb_policy_adam_set(self.h, _ptr(arrs[0]), _ptr(arrs[1]), int(step)), "policy_adam_set")

    def adam_get(self):
        m, v = np.empty(self.d, np.float32), np.empty(self.d, np.float32)
        step = C.c_int64()
        self._ck(self.lib.mjb_policy_adam_get(self.h, _ptr(m), _ptr(v), C.byref(step)), "policy_adam_get")
        return m, v, int(step.value)

    def bc_loss(self, loss):
        """Full-batch BC loss ("mle" or "mse") of theta_new over the resident batch."""
        out = C.c_double()
        self._ck(self.lib.mjb_policy_bc_loss(self.h, LOSS[loss], C.byref(out)), "policy_bc_loss")
        return float(out.value)

    def last_sgd_ms(self):
        """CUDA-event time of the last policy_sgd chain."""
        t = C.c_float()
        self._ck(self.lib.mjb_policy_sgd_timing(self.h, C.byref(t)), "policy_sgd_timing")
        return float(t.value)

    def set_tensor_cores(self, on=True):
        """Returns True when the tcgen05 FVP path is active for this policy shape."""
        return self.lib.mjb_policy_set_tensor_cores(self.h, int(on)) == 0 and bool(on)

    def last_vectors(self):
        g = np.empty(self.d, dtype=np.float32)
        x = np.empty(self.d, dtype=np.float32)
        self._ck(self.lib.mjb_policy_last_vectors(self.h, _ptr(g), _ptr(x)), "last_vectors")
        return g, x

    # ------------------------------------------------------------------ baseline
    def vf_set_state(self, w, m=None, v=None, step=-1):
        arrs = [None if a is None else _f32(a) for a in (w, m, v)]
        self._ck(self.lib.mjb_vf_set_state(self.h, *[_ptr(a) for a in arrs], int(step)), "vf_set_state")

    def vf_get_state(self):
        w, m, v = (np.empty(self.vf_d, dtype=np.float32) for _ in range(3))
        step = C.c_int64()
        self._ck(self.lib.mjb_vf_get_state(self.h, _ptr(w), _ptr(m), _ptr(v), C.byref(step)), "vf_get_state")
        return w, m, v, int(step.value)

    def vf_fit(self, perms, batch_size=64, lr=1e-3, reg_coef=0.0, return_errors=False):
        perms = np.ascontiguousarray(perms, dtype=np.int32)
        if perms.ndim == 1:
            perms = perms[None]
        err = (C.c_double * 2)()
        self._ck(self.lib.mjb_vf_fit(self.h, _ptr(perms), perms.shape[0], int(batch_size), float(lr), float(reg_coef),
                                     C.byref(err) if return_errors else None), "vf_fit")
        return (err[0], err[1]) if return_errors else None

    def vf_fit_begin(self, perms, batch_size=64, lr=1e-3, reg_coef=0.0, return_errors=False):
        perms = np.ascontiguousarray(perms, dtype=np.int32)
        if perms.ndim == 1:
            perms = perms[None]
        err = C.c_double()
        self._ck(self.lib.mjb_vf_fit_begin(self.h, _ptr(perms), perms.shape[0], int(batch_size), float(lr), float(reg_coef),
                                           C.byref(err) if return_errors else None), "vf_fit_begin")
        return err.value if return_errors else None

    def vf_fit_end(self, return_errors=False):
        err = C.c_double()
        self._ck(self.lib.mjb_vf_fit_end(self.h, C.byref(err) if return_errors else None), "vf_fit_end")
        return err.value if return_errors else None

    def vf_set_tensor_cores(self, on=True):
        """on: the single-SM tcgen05 fit kernel where the shape allows (default); off: the fp32-FMA kernel."""
        self._ck(self.lib.mjb_vf_set_tensor_cores(self.h, int(on)), "vf_set_tensor_cores")

    # ------------------------------------------------------------------ introspection
    def event_record(self, slot):
        self._ck(self.lib.mjb_event_record(self.h, int(slot)), "event_record")

    def event_elapsed_ms(self, a, b):
        t = C.c_float()
        self._ck(self.lib.mjb_event_elapsed_ms(self.h, int(a), int(b), C.byref(t)), "event_elapsed")
        return float(t.value)

    def kernel_launches(self):
        return int(self.lib.mjb_kernel_launches(self.h))

    def transfer_stats(self):
        """(h2d_bytes, d2h_bytes, uploads) issued by this engine so far -- counters kept by the library."""
        st = _native.TransferStats()
        self._ck(self.lib.mjb_transfer_stats(self.h, C.byref(st)), "transfer_stats")
        return int(st.h2d_bytes), int(st.d2h_bytes), int(st.uploads)

    def last_fit_ms(self):
        """CUDA-event time of the sequential Adam kernels of the last fit (joins a fit in flight)."""
        t = C.c_float()
        self._ck(self.lib.mjb_vf_fit_timing(self.h, C.byref(t)), "vf_fit_timing")
        return float(t.value)

    def last_fvp_ms(self):
        t = C.c_float()
        self.lib.mjb_fvp_timing(self.h, C.byref(t))
        return float(t.value)
