"""GAE(lambda) timings: `RolloutBuffer.gae` (include/hrl_b200.h `hrl_gae`, one launch) against the loop a user would write in
torch (reverse `for t in range(T)` with `torch.where`), and a check that both agree with a float64 run of that loop.

    python tools/gae_bench.py [--out FILE.json] [--reps 200]

Shapes (T, N) = (128, 4096) (the README's operating point), (2048, 256) (long horizon, few envs) and (128, 65536).  Data:
done with p = 0.05, the truncation bit on half of the dones, NaN in every terminal value that is not selected.
Timings are CUDA events, medians of 5 windows after a warm-up:
  - `kernel_l2_us`: back-to-back calls, so the buffers stay in L2 wherever they fit in its 126 MB - the state right after a
    rollout, which has just written them (the byte counts below say which shapes fit);
  - `kernel_cold_us`: a 256 MB write before every call evicts them first (events around the kernel only);
  - `torch_loop_us`: the torch loop, events around the whole call (host-bound: its launches are what the GPU waits for).
Bytes: `min_bytes` is what the computation has to move at least: per (t, e) rew 4 B, done 1 B, the flag of info[t, e, 2]
4 B, values 4 B, adv and ret 8 B; plus values[T] and the terminal values that are selected.  `kernel_l2_GBps` and
`kernel_cold_GBps` are min_bytes over the kernel time.  The card's name and power limit are recorded in the same run.
Needs a GPU; writes only --out."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = [(128, 4096), (2048, 256), (128, 65536)]
GAMMA, LAM = 0.99, 0.95
TOL = 1e-5


def make_buffer(T, N, seed=0):
    import torch
    from types import SimpleNamespace
    from hrl_pybullet_envs_b200 import config as K
    from hrl_pybullet_envs_b200.vec_env import RolloutBuffer
    g = torch.Generator(device="cuda").manual_seed(seed)
    buf = RolloutBuffer(SimpleNamespace(device=torch.device("cuda", 0), N=N, D=1, A=1, kind=K.HRL_ANT_FLAGRUN), T, info=True)
    u = lambda *s: torch.rand(*s, generator=g, device="cuda")                       # noqa: E731
    buf.done.copy_(u(T, N) < 0.05)
    trunc = buf.done & (u(T, N) < 0.5)
    buf.info[..., 2] = trunc.float() + 2.0 * (u(T, N) < 0.3).float()
    buf.rew.copy_(torch.randn(T, N, generator=g, device="cuda") + 5000.0 * (u(T, N) < 0.01).float())
    values = torch.randn(T + 1, N, generator=g, device="cuda") * 10
    tv = torch.randn(T, N, generator=g, device="cuda") * 10
    tv[~trunc] = float("nan")
    return buf, values, tv, trunc


def torch_gae(rew, done, values, tv, trunc, gamma, lam):
    """The loop a user writes: one reverse pass over T, every choice a torch.where."""
    import torch
    T = rew.shape[0]
    adv = torch.empty_like(rew)
    a = torch.zeros_like(rew[0])
    for t in reversed(range(T)):
        nxt = torch.where(done[t], torch.where(trunc[t], tv[t], 0.0), values[t + 1])
        delta = rew[t] + gamma * nxt - values[t]
        a = torch.where(done[t], delta, delta + gamma * lam * a)
        adv[t] = a
    return adv, adv + values[:T]


def scale(rew, done, values, tv, trunc, gamma, lam):
    """S_t = sum_{k >= t} (gamma lam)^(k - t) (|r_k| + gamma |next_k| + |V_k|) in float64 (tests/test_gpu_gae.py)."""
    import torch
    nxt = torch.where(done, torch.where(trunc, tv, 0.0), values[1:])
    m = (rew.abs() + gamma * nxt.abs() + values[:-1].abs()).double()
    S = torch.empty_like(m)
    s = torch.zeros_like(m[0])
    for t in reversed(range(m.shape[0])):
        s = m[t] + gamma * lam * s
        S[t] = s
    return S


def timed(fn, reps, windows=5):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out = []
    for _ in range(windows):
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1) * 1e3 / reps)
    return sorted(out)[windows // 2], out


def timed_cold(fn, reps, windows=5):
    """Events around fn() alone, with a 256 MB write (twice the L2) before every call."""
    import torch
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    out = []
    for _ in range(windows):
        for a, b in ev:
            flush.fill_(1.0)
            a.record()
            fn()
            b.record()
        torch.cuda.synchronize()
        out.append(sum(a.elapsed_time(b) for a, b in ev) * 1e3 / reps)
    return sorted(out)[windows // 2], out


def bench_shape(T, N, reps):
    import torch
    buf, values, tv, trunc = make_buffer(T, N)
    adv, ret = torch.empty_like(buf.rew), torch.empty_like(buf.rew)
    kernel = lambda: buf.gae(values, GAMMA, LAM, terminal_values=tv, out=(adv, ret))     # noqa: E731
    loop = lambda: torch_gae(buf.rew, buf.done, values, tv, trunc, GAMMA, LAM)           # noqa: E731
    for _ in range(20):
        kernel()
    loop()
    torch.cuda.synchronize()
    # agreement: both against the same loop in float64
    a64, r64 = torch_gae(buf.rew.double(), buf.done, values.double(), tv.double(), trunc, GAMMA, LAM)
    S = scale(buf.rew, buf.done, values, tv, trunc, GAMMA, LAM)
    a_t, r_t = loop()
    kernel()
    res = {"T": T, "N": N}
    for name, (a, r) in (("kernel", (adv, ret)), ("torch_loop", (a_t, r_t))):
        ea, er = (a.double() - a64).abs(), (r.double() - r64).abs()
        res[name + "_max_err_over_S"] = float((ea / S.clamp_min(1e-30)).max())
        res[name + "_within_tol"] = bool(torch.isfinite(a).all() and torch.isfinite(r).all() and (ea <= TOL * S).all()
                                         and (er <= TOL * (S + values[:T].double().abs())).all())
    n_sel = int(trunc.sum())
    res["min_bytes"] = T * N * 21 + 4 * N + 4 * n_sel
    res["fits_l2_126MB"] = res["min_bytes"] < 126e6
    res["kernel_l2_us"], res["kernel_l2_all"] = timed(kernel, reps)
    res["kernel_cold_us"], res["kernel_cold_all"] = timed_cold(kernel, min(reps, 50))
    n_loop = max(3, min(20, 20000 // T))
    res["torch_loop_us"], res["torch_loop_all"] = timed(loop, n_loop, windows=3)
    res["kernel_l2_GBps"] = res["min_bytes"] / res["kernel_l2_us"] / 1e3
    res["kernel_cold_GBps"] = res["min_bytes"] / res["kernel_cold_us"] / 1e3
    res["speedup_vs_torch_loop"] = res["torch_loop_us"] / res["kernel_l2_us"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=200)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("gae_bench.py needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    out = {"gpu": smi.stdout.strip().splitlines()[0] if smi.stdout.strip() else "unknown",
           "sms": torch.cuda.get_device_properties(0).multi_processor_count, "gamma": GAMMA, "lam": LAM, "shapes": []}
    print("gpu:", out["gpu"], flush=True)
    for T, N in SHAPES:
        r = bench_shape(T, N, a.reps)
        out["shapes"].append(r)
        print("T %5d N %6d  kernel %8.2f us (L2) %8.2f us (cold)  %7.1f / %7.1f GB/s of %.1f MB  torch loop %10.1f us  x%.0f  "
              "agree: kernel %s torch %s" % (T, N, r["kernel_l2_us"], r["kernel_cold_us"], r["kernel_l2_GBps"], r["kernel_cold_GBps"],
                                             r["min_bytes"] / 1e6, r["torch_loop_us"], r["speedup_vs_torch_loop"],
                                             r["kernel_within_tol"], r["torch_loop_within_tol"]), flush=True)
    s = json.dumps(out, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s)
    if not all(r["kernel_within_tol"] and r["torch_loop_within_tol"] for r in out["shapes"]):
        sys.exit("results disagree beyond the tolerance")


if __name__ == "__main__":
    main()
