"""Timings of population evaluation (hrl_evaluate_mlp) against the fused rollout it replaces, with the card's name, power
limit and SM clock read in the same run.  CUDA events around each call, medians over rounds that alternate the compared
calls, with the spread (min, max) of the per-round values.  Prints one JSON document and writes it to --out (if given).
  - headline: AntGather 4096 envs, H = 64, T = 1000 from reset(): evaluate_mlp with P = 256 members of 16 envs against
    rollout_mlp with one policy (its RolloutBuffer is about 0.9 GB);
  - the loop it replaces: 16 sequential rollout_mlp calls on 16-env handles against one evaluate_mlp at N = 256, P = 16;
  - PointGather: the headline at 4096 envs, and 16 sequential rollout_mlp calls on 256-env handles against one
    evaluate_mlp at N = 4096, P = 16;
  - no regression: rollout_mlp (want_info + want_terminal_obs) at 4096 AntGather envs, T = 32, on the library built from
    the parent commit (--parent-lib) and on this one, alternated in the same process.
Every timed call starts from reset(), which is outside the timed window."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
from hrl_pybullet_envs_b200 import RolloutBuffer, VecEnv, _cabi


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def timed_us(setup, fn):
    setup()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); fn(); b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3


def mlp(D, A, H=64, P=None, seed=0):
    g = torch.Generator().manual_seed(seed)
    lead = () if P is None else (P,)
    return tuple((((torch.rand(*lead, o, i, generator=g) * 2 - 1) * 0.3).cuda(), ((torch.rand(*lead, o, generator=g) * 2 - 1) * 0.1).cuda())
                 for o, i in ((H, D), (H, H), (A, H)))


def compare(calls, rounds, T):
    """calls: {name: (setup, fn)}, alternated round by round; per-step microseconds."""
    for s, f in calls.values():     # warm-up
        s(); f()
    torch.cuda.synchronize()
    per = {k: [] for k in calls}
    for _ in range(rounds):
        for k, (s, f) in calls.items():
            per[k].append(timed_us(s, f) / T)
    return {k: dict(median_us_per_step=float(np.median(v)), min=float(np.min(v)), max=float(np.max(v)), rounds=v) for k, v in per.items()}


def headline(env_id, N=4096, P=256, T=1000, rounds=7):
    vec = VecEnv(env_id, N, seed=1, max_episode_steps=T)
    members = mlp(vec.D, vec.A, P=P, seed=1)
    one = tuple((W[0], b[0]) for W, b in members)
    buf = RolloutBuffer(vec, T)
    out = (torch.empty(N, device="cuda"), torch.empty(N, dtype=torch.int32, device="cuda"), torch.empty(N, dtype=torch.bool, device="cuda"))
    res = compare({"evaluate_mlp_P%d" % P: (vec.reset, lambda: vec.evaluate_mlp(members, T, sigma=0.1, out=out)),
                   "rollout_mlp_P1": (vec.reset, lambda: vec.rollout_mlp(one, T, buf=buf, sigma=0.1))}, rounds, T)
    assert bool(out[2].all())
    gb = sum(t.numel() * t.element_size() for t in (buf.obs, buf.act, buf.rew, buf.done)) / 1e9
    return dict(env=env_id, N=N, P=P, H=64, T=T, rollout_buffer_GB=gb, **res)


def loop(env_id, P=16, M=16, T=1000, rounds=5):
    big = VecEnv(env_id, P * M, seed=1, max_episode_steps=T)
    shards = [VecEnv(env_id, M, seed=1, env_index_offset=m * M, max_episode_steps=T) for m in range(P)]
    members = mlp(big.D, big.A, P=P, seed=2)
    bufs = [RolloutBuffer(s, T) for s in shards]
    out = (torch.empty(P * M, device="cuda"), torch.empty(P * M, dtype=torch.int32, device="cuda"),
           torch.empty(P * M, dtype=torch.bool, device="cuda"))

    def reset_all():
        for s in shards:
            s.reset()

    def sequential():
        for m, s in enumerate(shards):
            s.rollout_mlp(tuple((W[m], b[m]) for W, b in members), T, buf=bufs[m], sigma=0.1)
    res = compare({"evaluate_mlp_N%d_P%d" % (P * M, P): (big.reset, lambda: big.evaluate_mlp(members, T, sigma=0.1, out=out)),
                   "%dx_rollout_mlp_N%d" % (P, M): (reset_all, sequential)}, rounds, T)
    return dict(env=env_id, P=P, M=M, H=64, T=T, **res)


def regression(parent_lib, env_id="AntGatherBulletEnv-v0", N=4096, T=32, rounds=9, reps=5):
    new = _cabi.lib()
    old = ctypes.CDLL(parent_lib)
    for s in _cabi.SYMBOLS:           # the parent's symbols (it lacks the new ones) with this build's signatures
        if hasattr(old, s):
            getattr(old, s).argtypes, getattr(old, s).restype = getattr(new, s).argtypes, getattr(new, s).restype
    envs = {}
    for name, L in (("parent", old), ("new", new)):
        _cabi._lib = L                # VecEnv binds the library loaded at construction
        try:
            envs[name] = VecEnv(env_id, N, seed=1)
        finally:
            _cabi._lib = new
    vec0 = envs["new"]
    layers = mlp(vec0.D, vec0.A)
    sig = torch.full((vec0.A,), 0.3, device="cuda")
    bufs = {k: RolloutBuffer(v, T, info=True, terminal_obs=True) for k, v in envs.items()}

    def run(k):
        for _ in range(reps):
            envs[k].rollout_mlp(layers, T, buf=bufs[k], sigma=sig, want_info=True, want_terminal_obs=True)
    calls = {k: (envs[k].reset, (lambda k=k: run(k))) for k in envs}
    res = compare(calls, rounds, T * reps)
    same = all(torch.equal(getattr(bufs["parent"], f), getattr(bufs["new"], f)) for f in ("obs", "act", "rew", "done", "info"))
    return dict(env=env_id, N=N, T=T, calls_per_round=reps, parent_lib=os.path.relpath(parent_lib, ROOT), same_buffers=same, **res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", help="libhrl_b200.so built from the parent commit (the no-regression line)")
    ap.add_argument("--out")
    a = ap.parse_args()
    torch.cuda.init()
    res = dict(card_name_power_limit_sm_clock_max_sm_clock=card(), device=torch.cuda.get_device_name(0))
    res["headline"] = headline("AntGatherBulletEnv-v0")
    res["loop"] = loop("AntGatherBulletEnv-v0")
    res["point_headline"] = headline("PointGatherBulletEnv-v0")
    res["point_loop"] = loop("PointGatherBulletEnv-v0", P=16, M=256)
    if a.parent_lib:
        res["no_regression"] = regression(os.path.abspath(a.parent_lib))
    res["card_after"] = card()
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
