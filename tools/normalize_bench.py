"""Timings of observation and reward normalization (CUDA events, medians after warm-up), with the card's name and power limit
read in the same run.  Prints one JSON document and writes it to the path given as the first argument (if any).
  - fused rollout (rollout_mlp, want_info + want_terminal_obs) with and without obs_norm, alternated in the same run:
    AntGather 4096 envs T = 32, PointGather 4096 envs T = 32;
  - hrl_obs_moments against its float64 torch equivalent at 128 x 4096 x 46;
  - hrl_reward_scale against the torch loop over T (float64 returns, as SB3) at (128, 4096) and (128, 16384).
The statistics buffers (at most 96 MB) are re-read every call, so they are largely L2-resident (126 MB): "warm" numbers."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
from hrl_pybullet_envs_b200 import RunningNormalizer, VecEnv


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def timed(fn, reps, warm=3):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e3)
    return float(np.median(ts)), ts


def mlp(D, A, H=64, seed=0):
    g = torch.Generator().manual_seed(seed)
    return tuple((((torch.rand(o, i, generator=g) * 2 - 1) * 0.3).cuda(), ((torch.rand(o, generator=g) * 2 - 1) * 0.1).cuda())
                 for o, i in ((H, D), (H, H), (A, H)))


def bench_rollout(env_id, N=4096, T=32, rounds=5, reps=5):
    vec = VecEnv(env_id, N, seed=1)
    norm = RunningNormalizer(vec)
    norm.update_obs(vec.reset())
    layers = mlp(vec.D, vec.A)
    from hrl_pybullet_envs_b200 import RolloutBuffer
    buf = RolloutBuffer(vec, T, info=True, terminal_obs=True)
    sig = torch.full((vec.A,), 0.3, device="cuda")
    plain = lambda: vec.rollout_mlp(layers, T, buf=buf, sigma=sig, want_info=True, want_terminal_obs=True)  # noqa: E731
    normed = lambda: vec.rollout_mlp(layers, T, buf=buf, sigma=sig, want_info=True, want_terminal_obs=True, obs_norm=norm)  # noqa: E731
    res = {"plain_us_per_step": [], "norm_us_per_step": []}
    for _ in range(rounds):                              # alternate the two in the same run
        res["plain_us_per_step"].append(timed(plain, reps)[0] / T)
        res["norm_us_per_step"].append(timed(normed, reps)[0] / T)
    p, q = np.median(res["plain_us_per_step"]), np.median(res["norm_us_per_step"])
    res.update(env=env_id, N=N, T=T, median_plain=p, median_norm=q, ratio_norm_over_plain=q / p)
    return res


def bench_obs_moments(M=128 * 4096, D=46, reps=20):
    x = torch.randn(M, D, device="cuda") * 3 + 1
    n = RunningNormalizer((1, D))
    k_us, _ = timed(lambda: n.update_obs(x), reps)
    mom = torch.zeros(1 + 2 * D, dtype=torch.float64, device="cuda")
    mom[0] = 1e-4; mom[1 + D:] = 1.0

    def torch_ref():
        xd = x.double()
        bv, bm = torch.var_mean(xd, 0, unbiased=False)
        count, mean, var = mom[0], mom[1:1 + D], mom[1 + D:]
        delta, tot = bm - mean, count + M
        new_mean = mean + delta * M / tot
        new_var = (var * count + bv * M + delta * delta * count * M / tot) / tot
        return new_mean.float(), (1.0 / torch.sqrt(new_var + 1e-8)).float()
    t_us, _ = timed(torch_ref, reps)
    return dict(M=M, D=D, bytes=M * D * 4, hrl_obs_moments_us=k_us, torch_float64_us=t_us, speedup=t_us / k_us,
                GBps_of_input=M * D * 4 / k_us / 1e3)


def bench_reward_scale(T, N, reps=10):
    rew = torch.randn(T, N, device="cuda")
    done = torch.rand(T, N, device="cuda") < 0.02
    n = RunningNormalizer((N, 1))
    out = torch.empty_like(rew)
    k_us, _ = timed(lambda: n.scale_rewards(rew, done, out=out), reps)
    R = torch.zeros(N, dtype=torch.float64, device="cuda")
    m = torch.tensor([1e-4, 0.0, 1.0], dtype=torch.float64, device="cuda")

    def torch_loop():
        nonlocal R
        count, mean, var = m[0], m[1], m[2]
        res = torch.empty_like(rew)
        for t in range(T):
            R = R * 0.99 + rew[t].double()
            bv, bm = torch.var_mean(R, unbiased=False)
            delta, tot = bm - mean, count + N
            mean = mean + delta * N / tot
            var = (var * count + bv * N + delta * delta * count * N / tot) / tot
            count = tot
            res[t] = torch.clamp(rew[t] * (1.0 / torch.sqrt(var + 1e-8)).float(), -10, 10)
            R = torch.where(done[t], torch.zeros_like(R), R)
        return res
    t_us, _ = timed(torch_loop, 3, warm=1)
    return dict(T=T, N=N, hrl_reward_scale_us=k_us, torch_loop_us=t_us, speedup=t_us / k_us)


def main():
    torch.cuda.init()
    res = dict(card=card(), device=torch.cuda.get_device_name(0))
    res["rollout"] = [bench_rollout("AntGatherBulletEnv-v0"), bench_rollout("PointGatherBulletEnv-v0")]
    res["obs_moments"] = bench_obs_moments()
    res["reward_scale"] = [bench_reward_scale(128, 4096), bench_reward_scale(128, 16384)]
    s = json.dumps(res, indent=1)
    print(s)
    if len(sys.argv) > 1:
        os.makedirs(os.path.dirname(os.path.abspath(sys.argv[1])), exist_ok=True)
        with open(sys.argv[1], "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
