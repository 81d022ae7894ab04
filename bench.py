#!/usr/bin/env python
"""Benchmark of the post-rollout NPG/TRPO/DAPG update path (BASELINE.json metric: train_step/s and FVP/s on a
1e6-timestep batch).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config cfg3] [--impl reference] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  A "step" = everything mjrl's train_step does after sampling
(algos/batch_reinforce.py:94-112): returns -> baseline predict -> GAE -> whitening -> VPG -> 10-iteration CG
over Fisher-vector products -> step (+ TRPO line search) -> surrogate/KL re-evaluation -> MLPBaseline.fit
(1 epoch of sequential minibatch Adam).  `value` times it with the trajectories already resident in HBM (CUDA
events on the engine's stream, max over ranks); `e2e` times the public drop-in API (TRPO.update_from_paths(paths))
from host float64 path dicts, host<->device copies included.  Strong scaling: the 1e6-timestep batch is sharded
by trajectory over the ranks; one NCCL all-reduce of the flat gradient and of every FVP result.

`--impl reference` (and the `cpu_baseline` object of the default arm) time the UNMODIFIED reference package
(aravindr93/mjrl imported through oracle/ref_shim.py from baseline/_ref; the oracle restatement only when no copy of
the reference is present) on the box's host cores, with the torch thread count calibrated on the box: the reference
arm times one step on the full batch plus bounded-sample steps, `cpu_baseline` a bounded sample.

The default line also carries `roofline_hbm`: the HBM-bound Fisher-vector product of the linear policy at
BASELINE.json's cfg5 shape (376-dim observations, 5e5 timesteps), measured in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import faulthandler

import numpy as np

faulthandler.enable()
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # name: obs, act, hidden, n_traj, horizon, algo            (BASELINE.json configs[0..4], SURVEY 8d)
    "cfg1": dict(obs=6, act=2, hidden=(32, 32), n_traj=5, horizon=50, algo="npg", name="point_mass NPG 32x32 5x50"),
    "cfg2": dict(obs=8, act=2, hidden=(64, 64), n_traj=100, horizon=1000, algo="npg", name="Swimmer-v3 NPG 64x64 1e5"),
    "cfg3": dict(obs=17, act=6, hidden=(128, 128), n_traj=1000, horizon=1000, algo="trpo",
                 name="HalfCheetah-v3 TRPO 128x128 1e6"),
    "cfg4": dict(obs=39, act=28, hidden=(256, 256), n_traj=1000, horizon=200, algo="dapg",
                 name="Adroit door-v0 DAPG 256x256 2e5"),
    "cfg5": dict(obs=376, act=17, hidden=(), n_traj=500, horizon=1000, algo="npg", name="Humanoid-v3 linear NPG 5e5"),
}
GAMMA, LAM, CG_ITERS, DAMPING = 0.995, 0.97, 10, 1e-4
NPG_STEP, KL_DIST = 0.05, 0.01
VF = dict(reg_coef=1e-3, batch_size=64, epochs=1, learn_rate=1e-3)


def make_paths(cfg, first, count, seed=0):
    """Deterministic synthetic trajectories (float64 like the sampler delivers); path i depends only on (seed, i)
    so a rank can build its own shard."""
    paths = []
    for i in range(first, first + count):
        rng = np.random.RandomState((seed * 1000003 + i) % (2 ** 31 - 1))
        T = cfg["horizon"]
        paths.append(dict(observations=rng.randn(T, cfg["obs"]), actions=rng.randn(T, cfg["act"]),
                          rewards=rng.randn(T), terminated=False))
    return paths


def flops_per_sample_fvp(cfg):
    sizes = (cfg["obs"],) + tuple(cfg["hidden"]) + (cfg["act"],)
    P = sum(a * b for a, b in zip(sizes[:-1], sizes[1:]))
    if len(cfg["hidden"]) == 0:
        return 4 * P
    return 10 * P - 4 * sizes[0] * sizes[1]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        late = False
        if not self.rows:                      # a timed region shorter than nvidia-smi's start-up (cfg1: 6 ms): take the first
            t0 = time.time()                   # sample it delivers, i.e. the clocks right after the region, and say so
            while not self.rows and time.time() - t0 < 1.5:
                time.sleep(0.02)
            late = True
        self.proc.terminate()
        sm, mx, reasons, pw = [], [], set(), []
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        out = {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
               "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}
        if late:
            out["note"] = "timed region shorter than the sampler's start-up: first sample taken right after it"
        return out


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], tflops_burst=d["bf16_tflops"], tflops_sustained=d["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, tflops_burst=1590.0, tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


# ======================================================================================= CPU reference arm
def _reference_or_port():
    """The real aravindr93/mjrl package (through oracle/ref_shim.py: $MJRL_REF -> /root/reference -> baseline/_ref, the
    offline `pip install --target` of the unmodified reference that travels to the GPU box) or, when no copy exists,
    the oracle restatement."""
    from oracle import ref_shim                 # the CPU baseline legs are the one place bench.py runs oracle/
    if ref_shim.available():
        return ref_shim.load(), "reference"
    return None, "port"


def cpu_reference_step_fn(cfg, n_traj_sample, capture=None):
    """Returns (step_fn, n_samples, kind): one post-rollout step (batch_reinforce.py:94-112: compute_returns ->
    compute_advantages -> train_from_paths -> baseline.fit) of the CPU reference on `n_traj_sample` trajectories."""
    import contextlib
    import io
    import torch
    R, kind = _reference_or_port()
    paths0 = make_paths(cfg, 0, n_traj_sample)
    demo = make_paths(cfg, 10 ** 6, max(1, n_traj_sample // 40)) if cfg["algo"] == "dapg" else None
    if kind == "reference":
        es = R.EnvSpec(cfg["obs"], cfg["act"], cfg["horizon"])
        pol = R.LinearPolicy(es, seed=500) if len(cfg["hidden"]) == 0 else R.MLP(es, hidden_sizes=cfg["hidden"], seed=500)
        torch.manual_seed(1)
        bl = R.MLPBaseline(es, **VF)
        kw = dict(FIM_invert_args={"iters": CG_ITERS, "damping": DAMPING}, save_logs=False)
        if cfg["algo"] == "trpo":
            agent = R.TRPO(None, pol, bl, kl_dist=KL_DIST, **kw)
        elif cfg["algo"] == "dapg":
            agent = R.DAPG(None, pol, bl, demo_paths=demo, kl_dist=KL_DIST, **kw)
        else:
            agent = R.NPG(None, pol, bl, normalized_step_size=NPG_STEP, **kw)
        if capture is not None:
            capture["policy"], capture["baseline"] = pol, bl

        def step():
            paths = [dict(p) for p in paths0]
            buf = io.StringIO()
            with contextlib.redirect_stdout(buf):        # trpo.py:117-118 prints one line per backtrack
                R.process_samples.compute_returns(paths, GAMMA)
                R.process_samples.compute_advantages(paths, bl, GAMMA, LAM)
                agent.train_from_paths(paths)
                bl.fit(paths)
            return {"backtracks": buf.getvalue().count("Backtracking")}

        def fvp_time(reps=3):
            obs = np.concatenate([p["observations"] for p in paths0])
            act = np.concatenate([p["actions"] for p in paths0])
            v = np.random.RandomState(1).randn(pol.d).astype(np.float32)
            agent.HVP(obs, act, v, DAMPING)
            t0 = time.time()
            for _ in range(reps):
                agent.HVP(obs, act, v, DAMPING)
            return (time.time() - t0) / reps
        return step, n_traj_sample * cfg["horizon"], kind, fvp_time

    from oracle import npg_oracle as O
    spec = O.PolicySpec(cfg["obs"], cfg["act"], cfg["hidden"])
    state = dict(theta=O.init_policy_params(spec, 500), vf=O.VFState(cfg["obs"], (128, 128), seed=1))

    def step():
        paths = [dict(p) for p in paths0]
        O.compute_returns(paths, GAMMA)
        O.compute_advantages(paths, lambda p: O.vf_predict(state["vf"], p), GAMMA, LAM)
        obs = np.concatenate([p["observations"] for p in paths])
        act = np.concatenate([p["actions"] for p in paths])
        adv = O.whiten(np.concatenate([p["advantages"] for p in paths]))
        gb = None
        if demo is not None:
            gb = O.dapg_batch(obs, act, adv, np.concatenate([p["observations"] for p in demo]),
                              np.concatenate([p["actions"] for p in demo]), 1.0, 0.95, 0.0)
        out = O.policy_update(spec, state["theta"], obs, act, adv, cfg["algo"], step_size=NPG_STEP, kl_dist=KL_DIST,
                              cg_iters=CG_ITERS, damping=DAMPING, dtype=torch.float32, autograd=True, grad_batch=gb)
        state["theta"] = out["new_params"]
        perm = [np.random.permutation(obs.shape[0]) for _ in range(VF["epochs"])]
        O.vf_fit_torch(state["vf"], paths, perm, VF["epochs"], VF["batch_size"], VF["learn_rate"], VF["reg_coef"])
        return {"backtracks": int(out.get("backtracks", 0))}

    def fvp_time(reps=3):
        obs = np.concatenate([p["observations"] for p in paths0])
        v = np.random.RandomState(1).randn(spec.d).astype(np.float32)
        O.fvp(spec, state["theta"], obs, v, DAMPING, torch.float32, autograd=True)
        t0 = time.time()
        for _ in range(reps):
            O.fvp(spec, state["theta"], obs, v, DAMPING, torch.float32, autograd=True)
        return (time.time() - t0) / reps
    return step, n_traj_sample * cfg["horizon"], kind, fvp_time


def pick_cpu_threads(cfg):
    """The reference is torch-on-CPU: intra-op threads are the only parallelism it has.  More threads is not faster on
    a many-core host (round 1: 64 threads were 2-4x slower than 8), so the thread count is calibrated on one FVP of a
    small sample and the fastest count is used for every timed step; the table is reported."""
    import torch
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (min(8, ncpu), 16, 32, ncpu // 2, ncpu) if 1 <= c <= ncpu})
    step, n, kind, fvp_time = cpu_reference_step_fn(cfg, max(2, 20000 // cfg["horizon"]))
    table = {}
    for c in cands:
        torch.set_num_threads(c)
        table[c] = fvp_time(reps=2)
    best = min(table, key=table.get)
    torch.set_num_threads(best)
    return best, {str(k): round(v, 4) for k, v in table.items()}


def run_reference(args, cfg, rank, world):
    if rank != 0:
        return
    threads, table = pick_cpu_threads(cfg)
    n_full = cfg["n_traj"]
    n_s = min(cfg["n_traj"], max(5, 50000 // cfg["horizon"]))       # bounded sample for the warm-up / extra steps
    step_s, n, kind, fvp_time = cpu_reference_step_fn(cfg, n_s)
    for _ in range(args.warmup):
        step_s()
    # timed region: ONE step on the full batch (no extrapolation) + (steps-1) steps on the bounded sample
    full_s, backtracks = None, None
    if not args.reference_sample_only:
        step_f, n_f, _, _ = cpu_reference_step_fn(cfg, n_full)
        t0 = time.time()
        r = step_f()
        full_s = time.time() - t0
        backtracks = r["backtracks"]
        del step_f
    k = args.steps - (full_s is not None)
    dt_s = None
    if k > 0:
        t0 = time.time()
        for _ in range(k):
            step_s()
        dt_s = (time.time() - t0) / k
    scale = (cfg["n_traj"] * cfg["horizon"]) / n
    sec_per_step = full_s if full_s is not None else dt_s * scale
    value = 1.0 / sec_per_step
    fvp_t = fvp_time() * scale
    if full_s is None:
        sample = "%d of %d trajectories (%d timesteps) per step; extrapolated linearly x%.0f" % (n_s, cfg["n_traj"], n, scale)
    else:
        sample = "1 timed step on the FULL batch (%d trajectories, %d timesteps, no extrapolation) = %.1f s" % (
            n_full, n_full * cfg["horizon"], full_s)
        if dt_s is not None:
            sample += ("; plus %d steps on %d trajectories (%d timesteps) = %.2f s each, x%.0f = %.1f s extrapolated "
                       "(cross-check only)" % (k, n_s, n, dt_s, scale, dt_s * scale))
    line = {"impl": "reference", "metric": "train_step_per_sec", "value": value, "unit": "train_step/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec_per_step * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(cfg, args, world), "fvp_per_sec": 1.0 / fvp_t,
            "trpo_backtracks_full_batch": backtracks,
            "cpu_baseline": {"value": value, "unit": "train_step/s", "cores": threads, "os_cpu_count": os.cpu_count(),
                             "kind": kind, "sample": sample, "thread_calibration_s_per_fvp": table,
                             "extrapolated_from_sample_ms": None if dt_s is None else dt_s * scale * 1e3},
            "e2e": {"value": value, "unit": "train_step/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def gpu_first_step_backtracks(cfg, n_traj_sample, cap):
    """First update_from_paths of the GPU engine on the CPU baseline's sample, from the reference objects' own initial
    policy parameters and baseline weights: returns the TRPO backtrack count (None for the other algorithms)."""
    if cfg["algo"] != "trpo":
        return None
    from mjrl_b200.algos.trpo import TRPO
    from mjrl_b200.baselines.mlp_baseline import MLPBaseline
    from mjrl_b200.policies.gaussian_mlp import MLP
    from mjrl_b200.utils.gym_env import EnvSpec
    es = EnvSpec(cfg["obs"], cfg["act"], cfg["horizon"])
    pol = MLP(es, hidden_sizes=cfg["hidden"], seed=500)
    pol.set_param_values(cap["policy"].get_param_values(), set_new=True, set_old=True)
    bl = MLPBaseline(es, **VF)
    bl.set_flat_weights(np.concatenate([p.data.numpy().ravel() for p in cap["baseline"].model.parameters()]))
    agent = TRPO(None, pol, bl, kl_dist=KL_DIST, FIM_invert_args={"iters": CG_ITERS, "damping": DAMPING})
    agent.verbose = False
    agent.update_from_paths([dict(p) for p in make_paths(cfg, 0, n_traj_sample)], GAMMA, LAM)
    return int(agent.last_step.backtracks)


def hbm_roofline_cfg5(peaks, reps=20):
    """The HBM-bound kernel of the path (SURVEY 8d: the north_star's HBM target is defined on cfg5): Fisher-vector
    product of the linear policy, 5e5 timesteps x 376 observations = 752 MB streamed once per launch (> L2)."""
    from mjrl_b200.engine import Engine
    c5 = CONFIGS["cfg5"]
    n = c5["n_traj"] * c5["horizon"]
    rng = np.random.RandomState(5)
    eng = Engine(c5["obs"], c5["act"], (), max_samples=n + 8, max_paths=c5["n_traj"] + 8)
    obs = rng.standard_normal((n, c5["obs"]))
    eng.upload_flat(obs, rng.standard_normal((n, c5["act"])), np.zeros(n), np.full(c5["n_traj"], c5["horizon"], np.int32),
                    np.zeros(c5["n_traj"], np.uint8))
    del obs
    theta = (0.01 * rng.standard_normal(eng.d)).astype(np.float32)
    theta[-c5["act"]:] = 0.0
    eng.set_params(theta)
    v = rng.standard_normal(eng.d).astype(np.float32)
    tc = bool(eng.set_tensor_cores(True))
    ms = []
    for i in range(reps + 3):
        eng.fvp(v, DAMPING)
        if i >= 3:
            ms.append(eng.last_fvp_ms())
    eng.close()
    t = float(np.mean(ms)) * 1e-3
    by = 4.0 * n * c5["obs"]
    prof = {}
    pj = os.path.join(ROOT, "profiles", "fvp_ncu_cfg5.json")
    if os.path.exists(pj):
        prof = json.load(open(pj))
    return {"bound": "hbm", "achieved": by / t / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
            "frac": by / t / 1e9 / peaks["hbm_gbs"], "traffic": prof.get("dram_bytes_per_launch"),
            "kernel": "linear_tc_kernel (tcgen05)" if tc else "linear_kernel<AG,MODE_FVP> (fp32 FMA)",
            "workload": c5["name"], "launch_ms": t * 1e3, "launch_ms_min": float(np.min(ms)), "launches_timed": reps,
            "algorithmic_bytes_per_launch": by, "peak_source": peaks["source"] + "; copy bandwidth",
            "note": "kernel timed alone (CUDA events on the engine stream around the launch); the 752 MB observation "
                    "matrix exceeds L2, so every launch streams it from HBM"}


def workload_config(cfg, args, world):
    return {"workload": cfg["name"], "obs_dim": cfg["obs"], "act_dim": cfg["act"], "hidden": list(cfg["hidden"]),
            "n_traj": cfg["n_traj"], "horizon": cfg["horizon"], "timesteps": cfg["n_traj"] * cfg["horizon"],
            "algo": cfg["algo"], "cg_iters": CG_ITERS, "damping": DAMPING, "vf_epochs": VF["epochs"],
            "parallelism": "dp%d (trajectory shards; every FVP ends in an all-reduce of d floats: fused peer-memory kernel over "
                           "NVLink when the ranks can map each other, else ncclAllReduce -- see fvp_allreduce; NCCL for the flat "
                           "gradient and the scalar statistics)" % world,
            "cache": "batch < L2 on purpose of the workload: obs stays L2-resident across the 10 CG FVPs of a step as in "
                     "production; every step also streams the 1e6-row fit gather + GAE arrays (> L2 in total)"}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, eng, st):
    """Write what the timed path computed in its last step, as its caller receives it, to out_dir/<name>.npy: the
    updated policy parameters, the step's vanilla and natural gradients and its statistics, the fitted baseline
    weights, and the per-timestep returns, baseline predictions, GAE advantages and whitened advantages of the
    resident batch (this rank's shard).  Every input is seeded, so two builds run with the same arguments can be
    compared array by array."""
    vpg, npg = eng.last_vectors()
    out = {"policy_params": eng.get_params(), "vpg_grad": vpg, "npg_grad": npg, "baseline_weights": eng.vf_get_state()[0],
           "returns": eng.returns(), "baseline": eng.baseline(), "advantages": eng.advantages(),
           "adv_white": eng.adv_white(),
           "step_stats": np.array([st.alpha, st.delta, st.kl_dist, st.surr_before, st.surr_after, st.vpg_dot_npg,
                                   st.backtracks, st.cg_iters_run], np.float64)}
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit("--dump-outputs: %d bytes of outputs exceed the %d-byte limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ======================================================================================= GPU arm
def run_gpu(args, cfg, rank, world, local_rank):
    import torch
    from mjrl_b200.algos.dapg import DAPG
    from mjrl_b200.algos.npg_cg import NPG
    from mjrl_b200.algos.trpo import TRPO
    from mjrl_b200.baselines.mlp_baseline import MLPBaseline
    from mjrl_b200.engine import DEMO
    from mjrl_b200.policies.gaussian_linear import LinearPolicy
    from mjrl_b200.policies.gaussian_mlp import MLP
    from mjrl_b200.utils.gym_env import EnvSpec
    from mjrl_b200 import runtime
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: mjrl_b200 has no CPU fallback (use --impl reference for the CPU arm)")

    # ---- shard by trajectory (contiguous ranges, strong scaling) ----
    per = [cfg["n_traj"] // world + (1 if r < cfg["n_traj"] % world else 0) for r in range(world)]
    first = sum(per[:rank])
    paths = make_paths(cfg, first, per[rank])
    n_local = per[rank] * cfg["horizon"]
    n_glob = cfg["n_traj"] * cfg["horizon"]
    # every rank is constructed with the SAME demonstration list; the agent keeps its shard (DAPG._local_demos)
    demo_all = make_paths(cfg, 10 ** 6, max(1, cfg["n_traj"] // 40)) if cfg["algo"] == "dapg" else None
    demo = None
    if demo_all is not None:
        from mjrl_b200.parallel import shard_paths
        demo = shard_paths(demo_all, world, rank) if world > 1 else demo_all

    es = EnvSpec(cfg["obs"], cfg["act"], cfg["horizon"])
    pol = LinearPolicy(es, seed=500) if len(cfg["hidden"]) == 0 else MLP(es, hidden_sizes=cfg["hidden"], seed=500)
    torch.manual_seed(1)
    bl = MLPBaseline(es, **VF)
    kw = dict(FIM_invert_args={"iters": CG_ITERS, "damping": DAMPING}, save_logs=False)
    if cfg["algo"] == "trpo":
        agent = TRPO(None, pol, bl, kl_dist=KL_DIST, **kw)
        agent.verbose = False            # the reference prints one line per backtrack; stdout carries the JSON line here
    elif cfg["algo"] == "dapg":
        agent = DAPG(None, pol, bl, demo_paths=demo_all, kl_dist=KL_DIST, **kw)
    else:
        agent = NPG(None, pol, bl, normalized_step_size=NPG_STEP, **kw)
    eng = agent._eng(n_local + (sum(len(p["actions"]) for p in demo) if demo else 0), len(paths))
    agent._push_policy(eng)
    bl._eng()

    def barrier():
        eng.synchronize()
        if dist is not None:
            dist.barrier()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---------------- value: inputs resident in HBM ----------------
    eng.upload_paths(paths)
    if demo:
        eng.upload_paths(demo, which=DEMO)
    step_args = dict(cg_iters=CG_ITERS, damping=DAMPING)
    if cfg["algo"] == "npg":
        step_args.update(step_size=NPG_STEP)
    else:
        step_args.update(step_size=KL_DIST, demo_lam=1.0)
    stats = []

    def device_step():
        eng.compute_returns(GAMMA)
        # host RNG draw, as optimize_model.py:22 (same values and RNG state as np.random.permutation(n) per epoch); the call
        # MLPBaseline.fit_begin makes: the NEXT step's draw is computed ahead on a worker thread and taken only if numpy's
        # global RNG state is still the one it started from (tests/test_perm_speculation.py)
        perm = runtime.global_permutations(n_glob, VF["epochs"])
        eng.vf_fit_begin(perm, VF["batch_size"], VF["learn_rate"], VF["reg_coef"])   # side stream: needs only the returns
        eng.vf_predict(prefit=True)           # pre-fit baseline, as in the reference's program order
        eng.compute_advantages(GAMMA, LAM)
        eng.process_paths()
        st = eng.step(cfg["algo"], **step_args)
        eng.vf_fit_end()
        stats.append(st)

    np.random.seed(0)
    for _ in range(args.warmup):
        device_step()
    del stats[:]
    barrier()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    launches0 = eng.kernel_launches()
    t_wall = time.time()
    eng.event_record(0)
    for _ in range(args.steps):
        device_step()
    eng.event_record(1)
    ms = eng.event_elapsed_ms(0, 1)
    barrier()
    wall = time.time() - t_wall
    launches = eng.kernel_launches() - launches0
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng, stats[-1])
    ms = max_over_ranks(ms)
    ms_per_step = ms / args.steps
    fvp_ms_kernel = float(np.mean([s.fvp_kernel_ms_sum / max(1, s.fvp_launches) for s in stats]))
    fit_steps = n_glob // VF["batch_size"] - 1
    fit_us = eng.last_fit_ms() * 1e3 / max(1, fit_steps * VF["epochs"])
    backtracks = [int(s.backtracks) for s in stats]
    phase = {k: float(np.mean([getattr(s, k) for s in stats])) for k in ("time_vpg_ms", "time_npg_ms", "time_eval_ms")}

    # ---------------- FVP/s: device-resident CG (10 x {FVP + all-reduce + fused update}) ----------------
    g = eng.vpg() if cfg["algo"] != "dapg" else eng.vpg(True, 1.0)
    eng.cg(g, iters=CG_ITERS, damping=DAMPING)
    eng.lib.mjb_policy_cg(eng.h, None, CG_ITERS, DAMPING, 0.0, None, 0, None)    # warm-up of exactly the timed call (graph capture)
    barrier()
    reps = 5
    eng.event_record(2)
    for _ in range(reps):
        eng.lib.mjb_policy_cg(eng.h, None, CG_ITERS, DAMPING, 0.0, None, 0, None)
    eng.event_record(3)
    cg_ms = max_over_ranks(eng.event_elapsed_ms(2, 3)) / reps
    fvp_per_sec = 1e3 / (cg_ms / CG_ITERS)

    # ---------------- e2e: public API from host float64 path dicts ----------------
    def e2e_step():
        fresh = [dict(p) for p in paths]                 # the dicts are re-populated; update_from_paths uploads per call
        agent.update_from_paths(fresh, GAMMA, LAM)

    e2e_warm = max(1, min(args.warmup, 3))
    e2e_steps = args.steps
    for _ in range(e2e_warm):
        e2e_step()
    barrier()
    tr0 = eng.transfer_stats()
    t0 = time.time()
    for _ in range(e2e_steps):
        e2e_step()
    barrier()
    e2e_s = max_over_ranks((time.time() - t0) / e2e_steps)
    tr1 = eng.transfer_stats()
    # bytes the ENGINE copied (library counters, mjb_transfer_stats), not a formula; uploads must equal the steps
    h2d = (tr1[0] - tr0[0]) / e2e_steps
    d2h = (tr1[1] - tr0[1]) / e2e_steps
    uploads = tr1[2] - tr0[2]
    expect_uploads = e2e_steps * (2 if demo else 1)
    if uploads != expect_uploads:
        raise SystemExit("e2e: %d trajectory uploads in %d steps (expected %d) -- the timed region skipped its H2D copy"
                         % (uploads, e2e_steps, expect_uploads))
    # trajectories as they cross PCIe: observations / actions rounded to fp32 while staging, rewards fp64
    min_h2d = n_local * ((cfg["obs"] + cfg["act"]) * 4 + 8)
    if h2d < min_h2d:
        raise SystemExit("e2e: %.0f B/step copied host->device, the trajectories alone are %d B" % (h2d, min_h2d))

    if rank != 0:
        runtime.shutdown()
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---------------- roofline of the dominant kernel (the FVP tile kernel) ----------------
    peaks = load_peaks()
    fl = flops_per_sample_fvp(cfg) * n_local
    by = 4.0 * n_local * cfg["obs"]
    linear = len(cfg["hidden"]) == 0
    t = fvp_ms_kernel * 1e-3
    if not t > 0:
        raise SystemExit("no FVP kernel timing was recorded inside the timed steps (fvp_kernel_ms = %r)" % fvp_ms_kernel)
    prof = {}
    pj = os.path.join(ROOT, "profiles", "fvp_ncu_%s.json" % args.config)
    if os.path.exists(pj) and world == 1:                # the ncu capture is of a 1-GPU launch: no traffic figure for a shard
        prof = json.load(open(pj))
    if linear:
        roof = {"bound": "hbm", "achieved": by / t / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": by / t / 1e9 / peaks["hbm_gbs"], "traffic": prof.get("dram_bytes_per_launch")}
    else:
        roof = {"bound": "tensor", "achieved": fl / t / 1e12, "peak": peaks["tflops_sustained"], "unit": "TFLOP/s",
                "frac": fl / t / 1e12 / peaks["tflops_sustained"], "traffic": prof.get("dram_bytes_per_launch")}
    sm_clock = (clk or {}).get("sm_mhz") or 1965.0
    fma_peak = 148 * 128 * 2 * sm_clock * 1e6 / 1e12
    tc_active = bool(eng.set_tensor_cores(True))
    if linear:
        kname = ("linear_tc_kernel (tcgen05 kind::f16, M=128 stacked fp16 hi/lo rows, TMEM-resident gradient accumulators)"
                 if tc_active else "linear_kernel<AG,MODE_FVP> (fp32 FMA)")
        if tc_active and cfg["obs"] % 4 == 0:
            kname = kname.replace("linear_tc_kernel", "linear_tc_tma_kernel (TMA-fed fp32 ring, warp-specialised)")
    else:
        kname = ("fvp_tc_kernel (tcgen05 kind::f16, two-term fp16 split = 3 MMAs per logical product, TMEM accumulators)"
                 if tc_active else "mlp_kernel<H,MT,MODE_FVP> (fp32 FMA)")
    roof.update({"kernel": kname,
                 "launch_ms": fvp_ms_kernel, "algorithmic_flops_per_launch": fl, "algorithmic_bytes_per_launch": by,
                 "peak_source": peaks["source"] + ("; bf16 dense sustained (kernel timed inside a long step)" if not linear else ""),
                 "hbm_frac": by / t / 1e9 / peaks["hbm_gbs"],
                 "fp32_fma_peak_tflops_at_observed_clock": fma_peak, "frac_of_fp32_fma_peak": fl / t / 1e12 / fma_peak,
                 "executed_tensor_flops_per_launch": (3 * fl if tc_active else 0),
                 "note": ("rank-0 shard; HBM-bound shape (SURVEY 8d): obs are streamed exactly once per launch; launch_ms"
                          if linear else "rank-0 shard; compute-bound shape (SURVEY 8d); launch_ms") + " is the mean CUDA-event time of the FVP launches "
                         "inside the timed steps, where the kernel shares the GPU with the concurrent baseline fit "
                         "(tensor-core fit kernel: 1 SM, FVP on 147; cluster fallback: 16 SMs); achieved counts ALGORITHMIC flops (10P-4P1 per timestep), not the 3x split MMAs"})

    # ---------------- CPU baseline (bounded sample, rank 0, N=1 only) ----------------
    cpu, bt_check, hbm = None, None, None
    if world == 1 and not args.no_cpu_baseline:
        threads, table = pick_cpu_threads(cfg)
        n_s = min(cfg["n_traj"], max(5, 100000 // cfg["horizon"]))
        cap = {}
        step, n, kind, fvp_time = cpu_reference_step_fn(cfg, n_s, capture=cap)
        # TRPO caveat (SURVEY 8d): the line search is data dependent -- same sample, same initial policy and baseline
        # on the GPU engine, backtrack counts of the first step must agree
        gpu_bt = gpu_first_step_backtracks(cfg, n_s, cap) if kind == "reference" else None
        r0 = step()
        if gpu_bt is not None:
            bt_check = {"sample_trajectories": n_s, "cpu_reference": int(r0["backtracks"]), "gpu": int(gpu_bt),
                        "equal": int(r0["backtracks"]) == int(gpu_bt)}
        t0 = time.time()
        reps_cpu = 2
        for _ in range(reps_cpu):
            step()
        dt = (time.time() - t0) / reps_cpu
        scale = n_glob / n
        cpu = {"value": 1.0 / (dt * scale), "unit": "train_step/s", "cores": threads,
               "os_cpu_count": os.cpu_count(), "kind": kind, "thread_calibration_s_per_fvp": table,
               "sample": "%d of %d trajectories (%d timesteps), %d timed steps after 1 warm-up; extrapolated linearly x%.0f"
                         % (n_s, cfg["n_traj"], n, reps_cpu, scale),
               "fvp_per_sec": 1.0 / (fvp_time() * scale)}
    if world == 1 and not args.no_hbm_roofline and args.config != "cfg5":
        runtime.shutdown()
        hbm = hbm_roofline_cfg5(peaks)

    line = {"metric": "train_step_per_sec", "value": 1e3 / ms_per_step, "unit": "train_step/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(cfg, args, world), "clocks": clk, "gpu_launches": int(launches),
            "e2e": {"value": 1.0 / e2e_s, "unit": "train_step/s", "ms_per_step": e2e_s * 1e3, "steps": e2e_steps,
                    "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "bytes_source": "mjb_transfer_stats counter deltas over the timed e2e steps (rank 0 shard)",
                    "uploads_in_timed_region": int(uploads),
                    "api": "mjrl_b200.algos.%s.update_from_paths(paths) on host float64 path dicts (per rank shard)"
                           % {"npg": "npg_cg.NPG", "trpo": "trpo.TRPO", "dapg": "dapg.DAPG"}[cfg["algo"]]},
            "fvp_per_sec": fvp_per_sec, "fvp_ms_in_cg": cg_ms / CG_ITERS, "fvp_kernel_ms": fvp_ms_kernel,
            "fvp_allreduce": ("none (1 rank)" if world == 1 else
                              "p2p (reduce + NVLink scatter + rank-ordered sum in one kernel)" if getattr(eng, "p2p", False)
                              else "nccl"),
            "wall_ms_per_step": wall / args.steps * 1e3, "phase_ms": phase, "trpo_backtracks": backtracks,
            "fit_us_per_adam_step": fit_us, "fit_adam_steps": fit_steps,
            "fit_permutation": "np.random.permutation stream, one draw per epoch and step; computed ahead of use on a host worker "
                               "thread and accepted only if numpy's global RNG state is unchanged (else drawn in place)",
            "roofline": roof, "roofline_hbm": hbm, "cpu_baseline": cpu, "trpo_backtrack_check": bt_check}
    print(json.dumps(line), flush=True)
    _exit_watchdog(60)
    runtime.shutdown()
    if dist is not None:
        dist.destroy_process_group()


def _exit_watchdog(seconds):
    """The result line is out; a teardown that does not finish (a peer rank died, a communicator that will not drain)
    must not keep the launcher waiting: end the process after `seconds`."""
    import threading
    t = threading.Timer(seconds, lambda: os._exit(0))
    t.daemon = True
    t.start()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="cfg3", choices=sorted(CONFIGS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-hbm-roofline", action="store_true", help="skip the cfg5 linear-policy FVP measurement")
    ap.add_argument("--reference-sample-only", action="store_true",
                    help="--impl reference: skip the full-batch step (bounded sample + extrapolation only)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the arrays the last timed step computed to DIR/<name>.npy (GPU arm, rank 0)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU arm")
    cfg = CONFIGS[args.config]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, cfg, rank, world)
        return
    run_gpu(args, cfg, rank, world, local_rank)


if __name__ == "__main__":
    main()
