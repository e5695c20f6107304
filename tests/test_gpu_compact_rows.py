"""The compact-row Ant kernel (ant_env_kernel<F, 0>: each solver row stored as its 8 non-zeros + the leg index, expanded
to 14 wide on load) is what hrl_create picks whenever it saves a wave of CTAs - 16 384 envs per B200 among others.
Every other oracle / golden test runs at N <= 4096, i.e. on the 14-wide kernel <F, 1>, so this file holds the compact
kernel to

  (a) the selection rule, observable through hrl_get_compact_rows;
  (b) the 14-wide kernel, one call at a time from bit-identical states: every family, every entry point, contact-heavy
      regimes, a ragged N and the production size;
  (c) the float64 oracle at 16 384 envs, with the tolerances and outlier rule of test_gpu_parity.test_one_step_parity;
  (d) the fused rollout, which always runs the 14-wide ROLL kernel, against step() on a compact handle.

Why (b) and (d) use the oracle tolerances and not bit equality: the solver arithmetic of the two variants is the same
(the expanded rows are the same floats, dot14 is packed fma2 / mul2 / add2 that the compiler cannot refold), but the two
template instantiations are contracted differently by the compiler elsewhere.  In leg_fk (hrl_ant.cuh:139, quaternion
to rotation matrix) one multiply + add pair is a fused FFMA in <F, 0> and an FMUL + FADD in <F, 1>
(profiles/compact_rows_contraction.txt, per-source-line instruction counts of both kernels).  So even hrl_observe, which
runs no physics, differs in the last bits from an identical state, and those bits are amplified by the solver like any
float32 rounding.  Every comparison therefore starts both handles from the same bits (get_state -> set_state), runs
ONE call, and holds the result to the tolerances the kernels are held to against the oracle.  A broken row layout
(wrong leg, lost right-hand side, idle rows not zeroed) moves nearly every env in contact far outside them."""
import time

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from hrl_pybullet_envs_b200 import config as K  # noqa: E402
from test_gpu_parity import POS_TOL, REW_TOL, VEL_TOL, _classify_outliers, _state_err  # noqa: E402

pytestmark = pytest.mark.gpu

FULL = 16384   # BASELINE config 5 (AntFlagrun) and the 8-GPU runs: envs per GPU


def _n_sm():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _rule(N, n_sm):
    """hrl_create's choice: compact iff 7 CTAs (of 8 envs) per SM need fewer waves than 6 do."""
    ctas = (N + 7) // 8
    return -(-ctas // (7 * n_sm)) < -(-ctas // (6 * n_sm))


def _compact(env):
    return env.L.hrl_get_compact_rows(env.h)


def _force(env, on):
    from hrl_pybullet_envs_b200 import _cabi
    _cabi.check(env.L.hrl_set_compact_rows(env.h, int(on)))
    assert _compact(env) == int(on)


def _pair(env_id, N, seed=3, **kw):
    """(compact, 14-wide) handles of the same config and seed."""
    from hrl_pybullet_envs_b200 import VecEnv
    a = VecEnv(env_id, N, seed=seed, **kw)
    b = VecEnv(env_id, N, seed=seed, **kw)
    _force(a, 1)
    _force(b, 0)
    return a, b


def _np(x):
    return x.cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


class _Cmp:
    """Compact handle `a` against 14-wide handle `b`, one call at a time from bit-identical states, with the tolerances and
    the outlier rule of test_gpu_parity.test_one_step_parity: an env is an outlier when its state leaves POS_TOL / VEL_TOL
    or its done flag / integer state differs (a contact or limit row switching on one sub-step apart, as against the
    oracle); outliers must stay below 5e-3 of the checked env-calls, every other env is held to the tolerances."""

    def __init__(self, env_id):
        self.env_id, self.checked, self.out = env_id, 0, 0
        self.worst = dict(pos=0.0, vel=0.0, obs=0.0, rew=0.0)
        self.sens_bad = self.sens_n = 0

    @staticmethod
    def sync(src, dst):
        f, i = src.get_state()
        dst.set_state(f, i)

    def _nsm(self, D):
        # Gather sector readings are discontinuous in the pose (an item on a bin edge flips bins): as in test_one_step_parity
        # only the continuous part is held to a tolerance, flipped readings must stay rare
        return 26 if self.env_id.startswith("AntGather") and D > 26 else D

    def check(self, what, a, b, outs=None):
        """Compare the states after one call; `outs` = ((obs, rew, done, info_raw, term), same for b) of a step."""
        fa, ia = a.get_state(); fb, ib = b.get_state()
        fa, fb, ia, ib = _np(fa), _np(fb), _np(ia), _np(ib)
        assert np.isfinite(fa).all() == np.isfinite(fb).all(), what
        ep, ev = _state_err(fa, fb)
        ok = (ep < POS_TOL) & (ev < VEL_TOL) & (ia == ib).all(axis=1)
        if outs is not None:
            (oa, ra, da, xa, ta), (ob, rb, db, xb, tb) = [[_np(v) if v is not None else None for v in o] for o in outs]
            da, db = da.astype(bool), db.astype(bool)
            ok &= da == db
            idx = np.nonzero(ok)[0]
            nsm = self._nsm(oa.shape[1])
            eo = float(np.abs(oa[idx, :nsm] - ob[idx, :nsm]).max(initial=0))
            assert eo < 2e-2, (what, eo)
            if nsm < oa.shape[1] and len(idx):
                self.sens_bad += int((np.abs(oa[idx, nsm:] - ob[idx, nsm:]) > 2e-3).sum()); self.sens_n += oa[idx, nsm:].size
            er = float(np.abs(ra[idx] - rb[idx]).max(initial=0))
            if not self.env_id.startswith("AntFlagrun"):   # Flagrun's progress reward amplifies 1e-3 m by 1/dt (as vs the oracle)
                assert er <= REW_TOL, (what, er)
            assert np.array_equal(xa[idx][:, 1:], xb[idx][:, 1:]), what   # dead_rew / goals_left, TimeLimit + goal flags, length
            fin = idx[da[idx]]
            if ta is not None and len(fin):
                # the state after the auto-reset says nothing about the step that ended the episode: its terminal
                # observation does, and one outside 5e-3 (test_one_step_parity's bound) makes the env an outlier
                ok[fin[np.abs(ta[fin, :nsm] - tb[fin, :nsm]).max(axis=1) >= 5e-3]] = False
            self.worst["obs"] = max(self.worst["obs"], eo); self.worst["rew"] = max(self.worst["rew"], er)
        self.worst["pos"] = max(self.worst["pos"], float(ep[ok].max(initial=0)))
        self.worst["vel"] = max(self.worst["vel"], float(ev[ok].max(initial=0)))
        self.checked += len(ok); self.out += int((~ok).sum())

    def finish(self, label):
        frac = self.out / max(self.checked, 1)
        print("%s: %d env-calls, worst pos %.2e vel %.2e obs %.2e rew %.2e, outliers %d (%.2e), flipped sector readings %d of %d"
              % (label, self.checked, self.worst["pos"], self.worst["vel"], self.worst["obs"], self.worst["rew"], self.out, frac,
                 self.sens_bad, self.sens_n))
        assert frac < 5e-3, (self.out, self.checked)
        assert self.sens_bad <= 2e-4 * max(self.sens_n, 1), (self.sens_bad, self.sens_n)


def _throw(envs, gen):
    """The thrown-ant state of tools/bounds_run.py, written into every handle: random orientation, z = 0.3, fast, aimed
    at the walls, Gather cubes right under the ants.  It drives the per-env contact and joint-limit row counts to their
    maximum and gives a warp envs with very different row counts, so idle solver visits happen."""
    f, i = envs[0].get_state()
    N, env_id = f.shape[0], envs[0].env_id
    q = torch.randn(N, 4, generator=gen, device="cuda")
    f[:, K.SF_QUAT:K.SF_QUAT + 4] = q / q.norm(dim=1, keepdim=True)
    f[:, K.SF_POS + 2] = 0.3
    half = 4.0 if "Maze" in env_id else 5.0
    f[:, K.SF_POS] = (torch.rand(N, generator=gen, device="cuda") * 2 - 1) * half
    f[:, K.SF_LINVEL:K.SF_LINVEL + 3] = torch.randn(N, 3, generator=gen, device="cuda") * 6
    f[:, K.SF_ANGVEL:K.SF_ANGVEL + 3] = torch.randn(N, 3, generator=gen, device="cuda") * 4
    if "Gather" in env_id:
        f[:, K.SF_ITEMS:K.SF_ITEMS + 32] = f[:, K.SF_POS:K.SF_POS + 2].repeat(1, 16) + torch.randn(N, 32, generator=gen, device="cuda") * 0.4
    for e in envs:
        e.set_state(f, i)


def _actions(regime, gen, N, A, t):
    a = torch.rand(N, A, generator=gen, device="cuda") * 2 - 1
    if regime == "saturated" or (regime == "thrown" and t % 3 == 0):
        a = torch.sign(a)   # joints driven onto their limits
    return a


def _actions(regime, gen, N, A, t):
    a = torch.rand(N, A, generator=gen, device="cuda") * 2 - 1
    if regime == "saturated" or (regime == "thrown" and t % 3 == 0):
        a = torch.sign(a)   # joints driven onto their limits
    return a


def _step_outs(ret, term=True):
    o, r, d, info = ret
    return o, r, d, info.raw, info["terminal_obs"] if term else None


def _drive(a, b, regime, T, label, seed=0):
    """T env steps (auto-reset, terminal observations) on the compact handle `a` and the 14-wide handle `b`, with
    substeps(1) / substeps(3), masked reset, observe and step_host interleaved.  Before every call b takes a's state bit
    for bit; after it both are compared (_Cmp).  Returns the in-kernel contact / limit-row counters of the window."""
    N, A = a.N, a.A
    cmp = _Cmp(a.env_id)
    gen = torch.Generator(device="cuda").manual_seed(seed)
    rng = np.random.default_rng(seed)
    a.reset(); cmp.sync(a, b)
    a.stats(reset=True); b.stats(reset=True)
    for t in range(T):
        if regime == "thrown" and t in (6, T // 2):
            _throw((a,), gen)
        act = _actions(regime, gen, N, A, t)
        cmp.sync(a, b)
        if t % 9 == 4:   # numpy in / numpy out (hrl_step_host)
            an = act.cpu().numpy()
            oa, ra, da, _ = a.step(an)
            outs_a = (oa.copy(), ra.copy(), da.copy(), a._info.clone(), None)
            ob, rb, db, _ = b.step(an)
            cmp.check("step_host t=%d" % t, a, b, (outs_a, (ob, rb, db, b._info, None)))
        else:
            outs_a = _step_outs(a.step(act, want_terminal_obs=True))
            cmp.check("step t=%d" % t, a, b, (outs_a, _step_outs(b.step(act, want_terminal_obs=True))))
        if t % 7 in (3, 5):
            n = 1 if t % 7 == 3 else 3
            cmp.sync(a, b)
            a.substeps(act, n); b.substeps(act, n)
            cmp.check("substeps(%d) t=%d" % (n, t), a, b)
        if t % 10 == 6:
            m = torch.tensor(rng.uniform(size=N) < 0.3, device="cuda")
            cmp.sync(a, b)
            oa = a.reset(m).clone()
            ob = b.reset(m)
            cmp.check("masked reset t=%d" % t, a, b)
            assert float((oa - ob)[:, :cmp._nsm(a.D)].abs().max()) < 2e-2, "masked reset t=%d obs" % t
        if t % 5 == 2:
            cmp.sync(a, b)
            oa = a.observe().clone()
            ob = b.observe()
            assert float((oa - ob)[:, :cmp._nsm(a.D)].abs().max()) < 2e-2, "observe t=%d" % t
    cmp.finish(label)
    sa, sb = a.stats(), b.stats()
    return sa, sb


# ------------------------------------------------------------------ (a) selection rule
def test_selection_rule_and_setter(monkeypatch):
    """hrl_get_compact_rows reports hrl_create's choice on either side of every wave boundary between 4096 and 16 384
    envs (computed here from the device's SM count), the setter flips it, and the kernels without compact rows (8 / 16
    lanes per env, PointGather) report 0."""
    from hrl_pybullet_envs_b200 import VecEnv, _cabi
    monkeypatch.delenv("HRL_B200_COMPACT", raising=False)
    n_sm = _n_sm()
    picks = {}
    for N in (4096, 7104, 7105, 8192, 8288, 8289, 12288, 16384):
        e = VecEnv("AntGatherBulletEnv-v0", N, seed=0)
        picks[N] = _compact(e)
        assert picks[N] == int(_rule(N, n_sm)), (N, n_sm, picks[N])
        _force(e, not picks[N])
        _force(e, picks[N])
        e.close()
    print("SMs %d, compact rows picked at:" % n_sm, picks)
    if n_sm == 148:   # B200: compact exactly in 7105..8288 and at 16 384 among these sizes
        assert [N for N, c in picks.items() if c] == [7105, 8192, 8288, 16384]
    e = VecEnv("AntFlagrunBulletEnv-v0", 64, seed=0)
    assert _compact(e) == 0
    _force(e, 1)
    for lanes in (8, 16):
        _cabi.check(e.L.hrl_set_lanes_per_env(e.h, lanes))
        assert _compact(e) == 0
    _cabi.check(e.L.hrl_set_lanes_per_env(e.h, 4))
    assert _compact(e) == 1
    p = VecEnv("PointGatherBulletEnv-v0", 64, seed=0)
    _cabi.check(p.L.hrl_set_compact_rows(p.h, 1))
    assert _compact(p) == 0
    monkeypatch.setenv("HRL_B200_COMPACT", "1")
    assert _compact(VecEnv("AntMjBulletEnv-v0", 64, seed=0)) == 1
    monkeypatch.setenv("HRL_B200_COMPACT", "0")
    assert _compact(VecEnv("AntMjBulletEnv-v0", FULL, seed=0)) == 0
    assert e.L.hrl_get_compact_rows(None) == -1 and e.L.hrl_set_compact_rows(None, 1) == -1


# ------------------------------------------------------------------ (b) compact against 14-wide, one call at a time
# the largest observations (Gather n_bins=16, Maze sense_target, Flagrun sensor) fill the task-layer tiles that alias the
# row buffer the most; Gather robot_coll_dist=0 runs the cube colliders and the contact pickup
CASES = [("AntGatherBulletEnv-v0", {}), ("AntGatherBulletEnv-v0", dict(n_bins=16)), ("AntGatherBulletEnv-v0", dict(robot_coll_dist=0)),
         ("AntMazeBulletEnv-v0", dict(sense_target=True)), ("AntMazeMjEnv-v0", {}), ("AntMjBulletEnv-v0", {}),
         ("AntFlagrunBulletEnv-v0", dict(use_sensor=True)), ("AntFlagrunBulletEnv-v0", {})]
CASE_IDS = ["%s-%s" % (e.replace("BulletEnv-v0", "").replace("Env-v0", ""), "+".join("%s=%s" % kv for kv in k.items()) or "default")
            for e, k in CASES]

# Floors of the in-kernel counters (contacts, limit rows per env-substep) over every case of a regime: about half the
# smallest value of the first B200 run (walk 0.91 / 0.98, saturated 0.83 / 1.15, thrown 0.29 / 1.84, printed by the
# tests), so that a regime cannot quietly stop producing contacts or limit rows.
STAT_FLOORS = {"walk": (0.45, 0.5), "saturated": (0.4, 0.55), "thrown": (0.15, 0.9)}


def _check_stats(label, regime, sa):
    print("%s: %.2f contacts, %.2f limit rows per env-substep" % (label, sa["contacts_per_substep"], sa["limit_rows_per_substep"]))
    c_min, l_min = STAT_FLOORS[regime]
    assert sa["contacts_per_substep"] >= c_min and sa["limit_rows_per_substep"] >= l_min, sa


@pytest.mark.parametrize("regime", ["walk", "saturated", "thrown"])
@pytest.mark.parametrize("env_id,kw", CASES, ids=CASE_IDS)
def test_compact_matches_wide(env_id, kw, regime):
    """N = 203 (a ragged last warp), both variants forced, 40 steps with resets inside the window (max_episode_steps=15)."""
    a, b = _pair(env_id, 203, max_episode_steps=15, **kw)
    label = "%s %s %s N=203" % (env_id, kw, regime)
    sa, _ = _drive(a, b, regime, 40, label, seed=len(regime))
    _check_stats(label, regime, sa)


def test_compact_matches_wide_capture_rollout():
    """A CUDA graph of one step captured on each variant (capture_rollout, with info), replayed from identical states."""
    from hrl_pybullet_envs_b200 import RolloutBuffer
    N = 203
    for env_id, kw in (("AntGatherBulletEnv-v0", dict(robot_coll_dist=0)), ("AntFlagrunBulletEnv-v0", dict(use_sensor=True))):
        a, b = _pair(env_id, N, max_episode_steps=3, **kw)
        cmp = _Cmp(env_id)
        a.reset(); cmp.sync(a, b)
        acts = torch.zeros(1, N, a.A, device="cuda")
        ga, bufa = a.capture_rollout(acts, RolloutBuffer(a, 1, info=True))
        gb, bufb = b.capture_rollout(acts, RolloutBuffer(b, 1, info=True))
        gen = torch.Generator(device="cuda").manual_seed(2)
        n_done = 0
        for rep in range(8):
            acts.copy_(torch.rand(1, N, a.A, generator=gen, device="cuda") * 2 - 1)
            cmp.sync(a, b)
            ga.replay(); gb.replay()
            torch.cuda.synchronize()
            cmp.check("%s replay %d" % (env_id, rep), a, b, ((bufa.obs[1], bufa.rew[0], bufa.done[0], bufa.info[0], None),
                                                            (bufb.obs[1], bufb.rew[0], bufb.done[0], bufb.info[0], None)))
            n_done += int(bufa.done[0].sum())
        cmp.finish("%s capture_rollout N=%d" % (env_id, N))
        assert n_done > 0


@pytest.mark.parametrize("env_id,regime", [("AntFlagrunBulletEnv-v0", "walk"), ("AntGatherBulletEnv-v0", "thrown")])
def test_compact_matches_wide_at_full_size(env_id, regime):
    """The production configuration itself: at 16 384 envs hrl_create picks the compact rows on a B200; 60 steps of it
    against a forced 14-wide handle, every entry point interleaved."""
    from hrl_pybullet_envs_b200 import VecEnv
    t0 = time.perf_counter()
    a = VecEnv(env_id, FULL, seed=5, max_episode_steps=25)
    b = VecEnv(env_id, FULL, seed=5, max_episode_steps=25)
    assert _compact(a) == int(_rule(FULL, _n_sm()))
    if _n_sm() == 148:
        assert _compact(a) == 1
    _force(a, 1)
    _force(b, 0)
    label = "%s %s N=%d" % (env_id, regime, FULL)
    sa, _ = _drive(a, b, regime, 60, label, seed=9)
    _check_stats(label, regime, sa)
    print("   wall time %.1f s" % (time.perf_counter() - t0))


# ------------------------------------------------------------------ (c) compact against the float64 oracle at 16 384
@pytest.mark.parametrize("env_id", ["AntGatherBulletEnv-v0", "AntFlagrunBulletEnv-v0"])
def test_compact_one_step_parity_full_size(env_id):
    """The checkpoint scheme of test_one_step_parity at N = 16 384 on the auto-selected (compact) kernel: copy the GPU
    state into the oracle, step both once; same tolerances, the same < 5e-3 outlier fraction, and every outlier must be
    explained by a discrete event of the oracle (_classify_outliers)."""
    from hrl_pybullet_envs_b200 import VecEnv
    from oracle import oracle as O
    t0 = time.perf_counter()
    N, T, EVERY = FULL, 96, 4   # 24 checkpoints: ~0.2-0.4 s of oracle each at threads=8 (printed below)
    g = VecEnv(env_id, N, device=0, seed=11)
    if _n_sm() == 148:
        assert _compact(g) == 1
    else:
        _force(g, 1)
    o = O.OracleVecEnv.make(env_id, N, seed=11, threads=8)
    g.reset(); o.reset()
    gen = torch.Generator().manual_seed(1)
    checked = n_out = 0
    worst_p = worst_v = worst_r = worst_o = 0.0
    sens_bad = sens_n = 0
    out_state, out_istate, out_act, out_ev, out_ep = [], [], [], [], []
    t_oracle = 0.0
    for t in range(T):
        a = torch.rand(N, g.A, generator=gen) * 2 - 1
        if t % EVERY:
            g.step(a.cuda())
            continue
        f, i = g.get_state()
        tt = time.perf_counter()
        o.set_state(f.cpu().numpy().astype(np.float64), i.cpu().numpy())
        oo, ro, do, io, to = o.step(a.numpy(), want_terminal=True)
        t_oracle += time.perf_counter() - tt
        og, rg, dg, info = g.step(a.cuda(), want_terminal_obs=True)
        f2, i2 = g.get_state(); fo, io2 = o.get_state()
        dg = dg.cpu().numpy(); rg = rg.cpu().numpy(); og = og.cpu().numpy()
        same = dg == do
        live = same & ~dg
        ep, ev = _state_err(f2.cpu().numpy()[live], fo[live])
        ok = (ep < POS_TOL) & (ev < VEL_TOL)
        n_out += int((~ok).sum()) + int((~same).sum())
        if (~ok).any():
            sel = np.nonzero(live)[0][~ok]
            out_state.extend(f.cpu().numpy()[sel].astype(np.float64)); out_istate.extend(i.cpu().numpy()[sel])
            out_act.extend(a.numpy()[sel]); out_ev.extend(ev[~ok].tolist()); out_ep.extend(ep[~ok].tolist())
        idx = np.nonzero(live)[0][ok]
        worst_p = max(worst_p, float(ep[ok].max(initial=0))); worst_v = max(worst_v, float(ev[ok].max(initial=0)))
        worst_r = max(worst_r, float(np.abs(rg[idx] - ro[idx]).max(initial=0)))
        if env_id == "AntGatherBulletEnv-v0":   # Flagrun's progress reward amplifies 1e-3 m by 1/dt (test_one_step_parity)
            assert np.abs(rg[idx] - ro[idx]).max(initial=0) <= REW_TOL
        nsm = 26 if env_id == "AntGatherBulletEnv-v0" else og.shape[1]   # Gather sector bins: see test_one_step_parity
        worst_o = max(worst_o, float(np.abs(og[idx, :nsm] - oo[idx, :nsm]).max(initial=0)))
        if nsm < og.shape[1] and len(idx):
            sens_bad += int((np.abs(og[idx, nsm:] - oo[idx, nsm:]) > 2e-3).sum()); sens_n += og[idx, nsm:].size
        fin = same & dg
        if fin.any():
            assert np.abs(info["terminal_obs"].cpu().numpy()[fin] - to[fin]).max() < 5e-3
            assert np.array_equal(i2.cpu().numpy()[fin], io2[fin])
        checked += int(live.sum())
    frac = n_out / max(checked, 1)
    print("%s N=%d compact: checked %d env-steps, worst pos %.2e vel %.2e rew %.2e obs %.2e, outliers %d (%.2e); oracle %.2e "
          "env-steps/s at threads=8" % (env_id, N, checked, worst_p, worst_v, worst_r, worst_o, n_out, frac,
                                        checked / max(t_oracle, 1e-9)))
    if out_ev:
        print("   outliers: max vel err %.3f, max pos err %.2e" % (max(out_ev), max(out_ep)))
        assert max(out_ev) < 3.0 and max(out_ep) < 2e-2
    if out_state:
        unexplained = _classify_outliers(env_id, np.array(out_state), np.array(out_istate), np.array(out_act))
        print("   outliers explained by a discrete event in the oracle: %d of %d" % (len(out_state) - unexplained, len(out_state)))
        assert unexplained == 0, (unexplained, len(out_state))
    assert checked > 0.9 * N * (T // EVERY)
    assert frac < 5e-3, (n_out, checked)
    assert worst_o < 2e-2
    assert sens_bad <= 2e-4 * max(sens_n, 1), (sens_bad, sens_n)
    print("   wall time %.1f s" % (time.perf_counter() - t0))


# ------------------------------------------------------------------ (d) fused rollout (14-wide ROLL) vs step() on compact
def _mlp(D, H, A, seed=0):
    g = torch.Generator().manual_seed(seed)

    def lin(o, i, s):
        return ((torch.rand(o, i, generator=g) * 2 - 1) * s).cuda(), ((torch.rand(o, generator=g) * 2 - 1) * 0.1).cuda()
    return (lin(H, D, 0.3), lin(H, H, 0.2), lin(A, H, 0.3))


ROLL_CASES = [("AntGatherBulletEnv-v0", 200, {}), ("AntMazeBulletEnv-v0", 200, dict(sense_target=True)), ("AntMazeMjEnv-v0", 200, {}),
              ("AntMjBulletEnv-v0", 200, {}), ("AntFlagrunBulletEnv-v0", 200, dict(use_sensor=True)),
              ("AntGatherBulletEnv-v0", FULL, {}), ("AntFlagrunBulletEnv-v0", FULL, {})]


@pytest.mark.parametrize("env_id,N,kw", ROLL_CASES)
def test_fused_rollout_matches_compact_step(env_id, N, kw):
    """A trainer that mixes rollout_mlp (always the 14-wide ROLL kernel) with step() on a compact handle: from identical
    states, one fused-rollout step and step() with the action it drew agree in obs, rew, done, info and terminal
    observations, 12 times in a row with auto-resets (5-step episodes).  N = 200 forces compact; N = 16 384 is compact by
    hrl_create's own choice on a B200."""
    from hrl_pybullet_envs_b200 import VecEnv
    a = VecEnv(env_id, N, seed=13, max_episode_steps=5, **kw)
    b = VecEnv(env_id, N, seed=13, max_episode_steps=5, **kw)
    if N == FULL and _n_sm() == 148:
        assert _compact(a) == 1 and _compact(b) == 1
    _force(b, 1)
    a.reset()
    layers = _mlp(a.D, 64, a.A)
    cmp = _Cmp(env_id)
    n_trunc = 0
    for t in range(12):
        cmp.sync(a, b)
        buf = a.rollout_mlp(layers, 1, sigma=0.2, noise_seed=4, want_info=True, want_terminal_obs=True)
        torch.cuda.synchronize()
        if t == 0:
            assert float((buf.obs[0] - b.observe())[:, :cmp._nsm(a.D)].abs().max()) < 2e-2
        outs_b = _step_outs(b.step(buf.act[0], want_terminal_obs=True))
        cmp.check("rollout step %d" % t, a, b, ((buf.obs[1], buf.rew[0], buf.done[0], buf.info[0], buf.terminal_obs[0]), outs_b))
        n_trunc += int(buf.truncated[0].sum())
    cmp.finish("%s %s N=%d rollout_mlp vs compact step" % (env_id, kw, N))
    assert n_trunc > 0
