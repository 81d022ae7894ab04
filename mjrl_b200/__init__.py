"""mjrl_b200 -- B200-native (sm_100a) engine for mjrl's post-rollout NPG / TRPO / DAPG update path, PPO-clip and
behaviour cloning.

Drop-in classes with the reference's names and signatures:
    mjrl_b200.algos.npg_cg.NPG, mjrl_b200.algos.trpo.TRPO, mjrl_b200.algos.dapg.DAPG
    mjrl_b200.algos.ppo_clip.PPO, mjrl_b200.algos.behavior_cloning.BC
    mjrl_b200.policies.gaussian_mlp.MLP, mjrl_b200.policies.gaussian_linear.LinearPolicy
    mjrl_b200.baselines.mlp_baseline.MLPBaseline
    mjrl_b200.utils.process_samples.compute_returns / compute_advantages, mjrl_b200.utils.cg_solve.cg_solve
All batched math runs in libmjrl_b200.so (hand-written CUDA behind the C ABI of include/mjrl_b200.h);
there is no CPU fallback."""
__version__ = "0.1.0"
