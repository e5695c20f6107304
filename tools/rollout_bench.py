"""Fused-rollout timings for training use, and an A/B of two builds of the library in one run.

    python tools/rollout_bench.py --parent-root OTHER_TREE [--reps 3] [--out FILE.json]

OTHER_TREE is another checkout of the project (e.g. the parent commit) with its library built; each build runs with its
own Python binding, selected by HRL_B200_LIB.  Alternates that build and this tree's build `--reps` times:
  - `bench.py --env AntGather`: config.policy_rollout.fused_rollout_us_per_step of each build;
  - a digest (sha256) of the default rollout buffers (obs / act / rew / done of 32 steps at 4096 AntGather envs, sigma 0.1)
    from the same seeded state: equal digests = the default path writes the same bytes.
This tree's build alone also times, at 4096 envs, 32 steps per launch:
  - AntGather (46-64-64-8 MLP): the default rollout against want_info + want_terminal_obs, alternating;
  - PointGather (18-64-64-2 MLP): the fused rollout against the same MLP in torch followed by step().
The working set (env state, weights, a 32-step buffer) fits in L2; nothing is flushed between launches.
The card's name and power limit are recorded in the same run.  Needs a GPU; writes only --out."""
import argparse
import hashlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _time_per_step(fn, T, launches=20, repeats=5):
    """µs per env step of `fn()` (one launch of T steps): median over `repeats` event-timed windows of `launches` calls."""
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out = []
    for _ in range(repeats):
        torch.cuda.synchronize()
        e0.record()
        for _ in range(launches):
            fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1) * 1e3 / (launches * T))
    return sorted(out)[len(out) // 2], out


def _layers(D, A, H=64, seed=7):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)

    def lin(o, i, sc):
        return ((torch.rand(o, i, generator=g, device="cuda") * 2 - 1) * sc, (torch.rand(o, generator=g, device="cuda") * 2 - 1) * 0.1)
    return (lin(H, D, 0.3), lin(H, H, 0.2), lin(A, H, 0.3))


def child(root, full):
    sys.path.insert(0, root)
    import torch
    from hrl_pybullet_envs_b200 import VecEnv, _cabi
    N, T = 4096, 32
    res = {"lib": os.environ["HRL_B200_LIB"], "version": _cabi.lib().hrl_version().decode()}
    env = VecEnv("AntGatherBulletEnv-v0", N, seed=0)
    env.reset()
    layers = _layers(env.D, env.A)
    buf = env.rollout_buffer(T)
    for i in range(10):                                 # land the ants (the bench's settle phase does the same)
        env.rollout_mlp(layers, T, buf=buf, sigma=0.1, noise_seed=i)
    env.rollout_mlp(layers, T, buf=buf, sigma=0.1, noise_seed=1)
    torch.cuda.synchronize()
    h = hashlib.sha256()
    for t in (buf.obs, buf.act, buf.rew, buf.done):
        h.update(t.cpu().numpy().tobytes())
    res["default_rollout_sha256"] = h.hexdigest()
    if full:
        ibuf = env.rollout_buffer(T)
        from hrl_pybullet_envs_b200 import RolloutBuffer
        tbuf = RolloutBuffer(env, T, info=True, terminal_obs=True)
        plain, extra = [], []
        for _ in range(5):                              # alternate the two variants
            plain.append(_time_per_step(lambda: env.rollout_mlp(layers, T, buf=ibuf, sigma=0.1, noise_seed=1), T, repeats=1)[0])
            extra.append(_time_per_step(lambda: env.rollout_mlp(layers, T, buf=tbuf, sigma=0.1, noise_seed=1, want_info=True,
                                                                want_terminal_obs=True), T, repeats=1)[0])
        res["antgather_4096"] = {"default_us_per_step": plain, "info_terminal_obs_us_per_step": extra,
                                 "finished_envs_per_step": float(tbuf.done.float().sum(1).mean())}
        env.close()
        p = VecEnv("PointGatherBulletEnv-v0", N, seed=0)
        p.reset()
        pl = _layers(p.D, p.A)
        pbuf = p.rollout_buffer(T)
        for i in range(3):
            p.rollout_mlp(pl, T, buf=pbuf, sigma=0.1, noise_seed=i)
        fused, fused_all = _time_per_step(lambda: p.rollout_mlp(pl, T, buf=pbuf, sigma=0.1, noise_seed=1), T)

        def torch_loop():
            o = p.observe()
            for _ in range(T):
                x = o
                for W, b in pl:
                    x = torch.tanh(torch.addmm(b, x, W.t()))
                o = p.step(x + 0.1 * torch.randn_like(x))[0]
        torch_loop()
        tl, tl_all = _time_per_step(torch_loop, T, launches=5)
        res["pointgather_4096"] = {"fused_rollout_us_per_step": fused, "fused_all": fused_all,
                                   "torch_mlp_plus_step_us_per_step": tl, "torch_all": tl_all,
                                   "policy": "%d-64-64-2 tanh MLP, sigma 0.1" % p.D, "steps_per_launch": T}
    print(json.dumps(res))


def _lib(root):
    return os.path.join(root, "hrl_pybullet_envs_b200", "libhrl_b200.so")


def run_bench(root, steps):
    env = dict(os.environ, HRL_B200_LIB=_lib(root))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "50",
                        "--env", "AntGather", "--skip-cpu"], env=env, capture_output=True, text=True, cwd=root)
    line = [l for l in r.stdout.splitlines() if l.startswith("{")]
    if r.returncode or not line:
        raise RuntimeError("bench.py failed in %s:\n%s" % (root, r.stderr[-3000:]))
    j = json.loads(line[-1])
    cfg = j.get("config", j)
    return cfg["policy_rollout"]["fused_rollout_us_per_step"], j.get("value")


def run_child(root, full):
    env = dict(os.environ, HRL_B200_LIB=_lib(root))
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", "--root", root] + (["--full"] if full else []),
                       env=env, capture_output=True, text=True)
    if r.returncode:
        raise RuntimeError("child failed in %s:\n%s" % (root, r.stderr[-3000:]))
    return json.loads(r.stdout.strip().splitlines()[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-root")
    ap.add_argument("--root", default=ROOT)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--bench-steps", type=int, default=640)
    ap.add_argument("--out", default=None)
    ap.add_argument("--child", action="store_true")
    ap.add_argument("--full", action="store_true")
    a = ap.parse_args()
    if a.child:
        return child(a.root, a.full)
    if not a.parent_root or not os.path.exists(_lib(a.parent_root)):
        sys.exit("--parent-root: another checkout with its library built, to compare against")
    parent = os.path.abspath(a.parent_root)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    out = {"gpu": smi.stdout.strip().splitlines()[0] if smi.stdout.strip() else "unknown", "parent_root": parent, "new_root": ROOT,
           "bench_fused_us_per_step": {"parent": [], "new": []}, "bench_value": {"parent": [], "new": []}, "digest": {}}
    for rep in range(a.reps):
        for tag, root in (("parent", parent), ("new", ROOT)):
            us, val = run_bench(root, a.bench_steps)
            out["bench_fused_us_per_step"][tag].append(us)
            out["bench_value"][tag].append(val)
            print(tag, rep, "fused us/step", us, "value", val, flush=True)
    for tag, root in (("parent", parent), ("new", ROOT)):
        r = run_child(root, full=(tag == "new"))
        out["digest"][tag] = r.pop("default_rollout_sha256")
        out.setdefault("child", {})[tag] = r
    out["default_rollout_bytes_equal"] = out["digest"]["parent"] == out["digest"]["new"]
    s = json.dumps(out, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s)


if __name__ == "__main__":
    main()
