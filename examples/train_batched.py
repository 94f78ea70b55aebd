"""The reference's own training loop (run.run_sequential) on the B200 stack: batched runner over the CUDA env, fused u8
observation front end, device epsilon-greedy, device learner.  MAC, agent network and replay buffer are the reference's.

    python baseline/fetch_ref.py                 # once, where the reference is mounted (copies it to baseline/_ref/)
    python examples/train_batched.py [envs] [env_steps] [--episode-stats] [--reward-shaping alpha,beta[,decay,prosocial]]

--episode-stats turns on the env's per-agent episode counters (extra_args episode_stats) and prints the social metrics they
give: efficiency, sustainability and peace, next to the collective return and equality.
--reward-shaping trains on the inequity-averse / prosocial shaped reward (extra_args reward_shaping; decay defaults to
0.99 * 0.975, prosocial to 0) and prints the mean shaped return next to the extrinsic statistics, which stay as they are.

Equivalent to adding these lines to the reference's registries (INTEGRATION.md section 6) and running
`python src/main.py --config=homophily --env-config=cleanup with runner=batched batch_size_run=256 ...`.
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from baseline import refloop  # noqa: E402

argv = sys.argv[1:]
shaping = None
if "--reward-shaping" in argv:
    i = argv.index("--reward-shaping")
    vals = [float(x) for x in argv[i + 1].split(",")]
    shaping = dict(zip(("alpha", "beta", "decay", "prosocial"), vals))
    del argv[i:i + 2]
episode_stats = "--episode-stats" in argv
argv = [a for a in argv if a != "--episode-stats"]
B = int(argv[0]) if len(argv) > 0 else 256
t_max = int(argv[1]) if len(argv) > 1 else 10 * B * 100
env_args = dict(num_agents=3, map="default3")
extra = {}
if episode_stats:
    extra["episode_stats"] = True
if shaping:
    extra["reward_shaping"] = shaping
if extra:
    env_args["extra_args"] = extra
cfg = refloop.load_config("cleanup", seed=0, use_cuda=True, save_model=False, t_max=t_max,
                          runner="batched", batch_size_run=B, buffer_size=max(B, 1024), buffer_cpu_only=False,
                          fused_frontend=True, action_selector="epsilon_greedy_b200", learner="homophily_learner_b200",
                          test_nepisode=B, test_interval=t_max, log_interval=B * 100, runner_log_interval=B * 100,
                          learner_log_interval=B * 100, env_args=env_args)
r = refloop.run_training(cfg, backend="b200", log_level="INFO")
steps = (t_max // (B * 100) + 1) * B * 100
print(f"{steps} env steps in {r['seconds']:.1f} s = {steps / r['seconds']:.0f} env-steps/s")
keys = ("return_mean", "collective_return_mean", "equality_metric_mean")
if episode_stats:
    keys += ("efficiency_mean", "sustainability_mean", "peace_mean", "apples_mean", "fires_mean", "hits_mean", "cleaned_mean")
if shaping:
    keys += ("shaped_return_mean",)
for k in keys + ("loss_value_env", "loss_value_inc", "loss_sim", "epsilon"):
    if k in r["stats"]:
        print(f"  {k}: {r['stats'][k]:.4f}")
