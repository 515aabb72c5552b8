"""The env step inside the fused policy rollouts (K5 `roboy_policy_rollout`, K6 `roboy_policy_rollout_tc` in its "tc" and
"tc_exact" modes) under every env flag, on MSJ and on MSJ-shaped robots with other limits, and at the band around the
bounds of reward_range.

The three kernels reach RoboyEnv.step through `sample_and_step` (policy_common.cuh), a copy of the step kernel's (K1)
arithmetic with the flags as run-time branches.  On an MSJ-shaped robot with other limits it divides by the spans in IEEE
division, where K1 uses the division checked on the device.  Only the env outputs are asserted here, which are exact by
design.  Each case runs one rollout on a prepared population: step counters spread over 1..400 with a cluster at the
timeout, injected held states (some infeasible, some with velocities far outside the velocity space), goals planted on
both sides of the reached threshold around the state each env reaches at a step k of the launch, and a policy shaped so
that part of the env-steps hold.  The rollout is then replayed three times on the clipped actions it stored:
  * on the CPU oracle: obs / done / goals / step words / error word and first offender exact, rewards to 1e-6, the
    statistics delta within the bound of test_gpu_episode_stats;
  * on K1 (`step_fused`, T calls) of a second handle restored from the snapshot: everything bit for bit, rewards included;
  * on a third, independent implementation: MSJ through the generic step kernel (rewards to PENALTY_REL), an
    MSJ-shaped robot with other limits on K1 kept on IEEE division (bit for bit).
"""
import ctypes
import math

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from test_gpu_episode_stats import K1_FLAGS, Tally, check_outputs, check_state, inject_held, make, policy_m, set_phases
from test_gpu_generic_robots import MSJ_SHAPED_OTHER_LIMITS, PENALTY_REL, environ, rewards_agree

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
MODES = ("fp32", "tc", "tc_exact")
ROBOTS = dict(msj=None, **MSJ_SHAPED_OTHER_LIMITS)
FLAG_IDS = ["default", "penalty", "nobonus", "manual_reset", "penalty_nobonus_manual"]
COUNTS = [k for k in orc.STAT_NAMES if k != "sum_reward"]


def hold_interval(bounds):
    """The float32 interval of actions whose rescale the Stub holds at (the same on every tendon of an MSJ-shaped robot)."""
    from gym_roboy_b200 import _native
    lib = _native.load()
    cfg = _native.RoboyCfg()
    _native.check(lib.roboy_cfg_msj(ctypes.byref(cfg)))
    for k, v in (bounds or {}).items():
        setattr(cfg, k, v)
    lo, hi = ctypes.c_float(), ctypes.c_float()
    _native.check(lib.roboy_hold_interval(ctypes.byref(cfg), ctypes.byref(lo), ctypes.byref(hi)))
    return lo.value, hi.value


def hold_policy(name, nan=False):
    """A policy whose actions hold on part of the env-steps, so that one launch has both branches.  The pi network is
    zero, so the mean is its output bias b3 exactly; components 1..7 have a tiny std.
      * MSJ, symmetric, asymmetric: b3 = the hold action, std[0] = half the width of the hold interval.
      * one-sided (hold centre -1): b3 = -3 on components 1..7, which clip to exactly -1; component 0 has mean -1 and
        std 0.01, so about half its samples clip to -1 and the env holds.
    `nan`: one NaN output bias, so that every action is NaN in that component (the action error, roboy_env.py:52).
    Returns (setup, exact16): exact16 says whether float16 carries b3, as the fast "tc" mode needs for these holds."""
    b = ROBOTS[name] or {}
    lo, hi = hold_interval(b)
    if name == "one_sided":
        head = np.full(8, -3.0, np.float32)
        head[0], std0 = -1.0, 1e-2
    else:
        head, std0 = orc.hold_action(b)[0], (hi - lo) / 2
    assert lo <= head[0] <= hi or name == "one_sided"

    def setup(policy):
        with torch.no_grad():
            for p_ in policy.pi.parameters():
                p_.zero_()
            policy.pi[4].bias.copy_(torch.as_tensor(head))
            policy.log_std.fill_(-40.0)
            policy.log_std[0] = math.log(std0)
            if nan:
                policy.pi[4].bias[5] = float("nan")
    return setup, bool((head.astype(np.float16).astype(np.float32) == head).all())


def plant_goals(client, ora, rng, seed, T, held, midpoints):
    """Goals at the threshold distance (x (1 -+ 1e-7), 0.7, 1.2) from the state each env is in after a step k of the
    launch, k drawn per env from 1..T: an env that does not hold samples orc.draw_state(seed, gid, counter + k)
    whatever the action.  Around their injected state for the held-state envs, and around the zero state for 10 % of the
    others: those reach their goal on a step where they hold.  `midpoints`: 10 % of the goals at the midpoint of the
    angle space (a division numerator of exactly zero)."""
    J, n = ora.J, ora.n
    lo, hi = ora.bounds["angle_low"], ora.bounds["angle_high"]
    gids = np.arange(n, dtype=np.uint64) + np.uint64(ora.cfg.env_id_base)
    k = rng.integers(1, T + 1, n)
    q = np.zeros((n, J))
    for kk in range(1, T + 1):
        sel = np.flatnonzero(k == kk)
        q[sel] = orc.draw_state(seed, gids[sel], ora.counter + kk, lo, hi, J=J)[0]
    zero = rng.random(n) < 0.1
    q[zero] = 0.0
    q[held] = ora.held[:J, held].T
    d = rng.normal(size=(n, J))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    thr_a, _ = orc.thresholds(ora.cfg)
    r = float(thr_a) * (1 + rng.choice([-1e-7, 1e-7, -0.3, 0.2], n))
    g = np.clip(q + d * r[:, None], lo, hi).astype(np.float32)
    if midpoints:
        g[rng.random(n) < 0.1] = ((lo.astype(np.float64) + hi.astype(np.float64)) / 2).astype(np.float32)
    client.set_goal(g)
    ora.goal[:] = g.T


class Rollout:
    """A handle of robot `name` with its oracle and a fused-rollout collector, the population prepared and snapshotted.
    `f64`: the handle is created (and given its reward range) under ROBOY_B200_PENALTY_F64=1."""

    def __init__(self, name, flags, mode, ept=0, n=6001, T=8, seed=29, env_id_base=0, setup=None, f64=False):
        from gym_roboy_b200.rollout import MlpPolicy, RolloutCollector
        self.name, self.flags, self.mode, self.ept, self.n, self.T = name, flags, mode, ept, n, T
        self.seed, self.env_id_base, self.f64 = seed, env_id_base, f64
        with environ(ROBOY_B200_PENALTY_F64="1" if f64 else "0"):
            env, self.client, self.ora = make(n, seed, ROBOTS[name], env_id_base=env_id_base, **flags)
            torch.manual_seed(0)
            policy = MlpPolicy().to(DEV)
            with torch.no_grad():
                policy.log_std.copy_(torch.linspace(-1.0, 0.7, 8))
            if setup is not None:
                setup(policy)
            self.col = RolloutCollector(env, policy, n_steps=T, fused=mode, noise_seed=5, envs_per_thread=ept)
        self.ora.reset()
        assert self.client.msj_kernels and self.client.penalty_float32 == (not f64 and name in ("msj", "symmetric"))
        rng = np.random.default_rng(seed)
        steps = rng.integers(1, 401, n)
        cluster = rng.random(n) < 0.2
        steps[cluster] = rng.integers(395, 401, int(cluster.sum()))   # timeouts inside the launch
        set_phases(self.client, self.ora, steps)
        held = np.sort(rng.choice(n, max(n // 50, 1), replace=False))
        feasible = rng.random(held.size) < 0.5
        inject_held(self.client, self.ora, rng, held, feasible)
        # velocities of 10 on every third held state leave MSJ's reward_range under the penalty; 1000 on the next third
        # leave that of every robot here
        J, fast = self.ora.J, held[1::3]
        q, qd = self.ora.held[:J, fast].T.copy(), np.full((fast.size, J), 1e3, np.float32)
        self.client.set_state(q, qd, feasible[1::3].astype(np.uint8), idx=fast)
        self.ora.held[J:, fast] = qd.T
        plant_goals(self.client, self.ora, rng, seed, T, held, midpoints=name != "msj")
        self.sd = self.client.state_dict()
        self.obs0 = self.col.obs[0].clone()

    def collect(self):
        self.col.collect()
        torch.cuda.synchronize()

    def restore(self):
        self.client.load_state_dict(self.sd)
        self.col.obs[0].copy_(self.obs0)

    def twin(self, **env):
        """Another handle of the same robot, seed and flags (created under the environment variables `env`), restored
        from the snapshot."""
        with environ(**env):
            _, c, _ = make(self.n, self.seed, ROBOTS[self.name], env_id_base=self.env_id_base, **self.flags)
        c.load_state_dict(self.sd)
        return c


def errors_equal(a, b):
    """(error word, first offending env): the first offender matters only where the word is set."""
    return a[0] == b[0] and (a[0] == 0 or a[1] == b[1])


def same_env_state(c1, c2):
    assert torch.equal(c1.goal, c2.goal) and torch.equal(c1.step_flags, c2.step_flags)
    assert errors_equal(c1.errors(), c2.errors()), (c1.errors(), c2.errors())
    s1, s2 = c1.stats(), c2.stats()
    for k in COUNTS:
        assert s1[k] == s2[k], (k, s1[k], s2[k])


def bitwise(r1, r2):
    return torch.equal(r1.view(torch.int32), r2.view(torch.int32))


def replay_on_step_kernel(client, col, T, same_reward):
    """T calls of the fused step on the clipped actions the rollout stored: the same outputs, step by step."""
    for t in range(T):
        client.step_fused(torch.clamp(col.actions[t], -1.0, 1.0).contiguous())
        assert torch.equal(client.obs, col.obs[t + 1]), ("obs", t)
        assert torch.equal(client.done_u8, col.dones[t]), ("done", t)
        assert same_reward(client.reward, col.rewards[t]), ("reward", t)


def run_case(name, flags, mode, ept=0, n=6001, T=8, env_id_base=0, nan=False):
    setup, exact16 = hold_policy(name, nan)
    r = Rollout(name, flags, mode, ept, n, T, env_id_base=env_id_base, setup=setup)
    client, ora, col = r.client, r.ora, r.col
    m, sel, _ = policy_m(client, mode, ept, T)
    tally = Tally(client, ora)
    r.collect()

    # ---- the CPU oracle on the clipped actions ----
    acts = np.clip(col.actions.cpu().numpy(), -1.0, 1.0)
    obs, rew, done = col.obs.cpu().numpy(), col.rewards.cpu().numpy(), col.dones.cpu().numpy()
    holds = ora.stats()["holds"]
    for t in range(T):
        o, rr, d = ora.step(acts[t])
        check_outputs(obs[t + 1], rew[t], done[t], o, rr, d, t)
    holds = ora.stats()["holds"] - holds
    check_state(client, ora)
    assert errors_equal(client.errors(), ora.errors()), (client.errors(), ora.errors())
    tally.check(col.rewards, m)
    if not nan and (mode != "tc" or exact16):
        assert 0 < holds < n * T, holds
        if flags.get("penalty"):
            assert client.errors()[0] & orc.ERR_REWARD_RANGE   # the held velocities of 1000 leave reward_range
    assert ora.stats()["episodes"] > 0

    # ---- K1 on a second handle: bit for bit (other limits: IEEE division in K5 / K6, checked fast division in K1) ----
    k1 = r.twin()
    assert k1.msj_kernels and k1.fast_division
    replay_on_step_kernel(k1, col, T, bitwise)
    same_env_state(k1, client)
    k1.close()

    # ---- an independent implementation on a third handle ----
    if name == "msj":
        other = r.twin(ROBOY_B200_FORCE_GENERIC="1")
        assert not other.msj_kernels
        penalty = bool(flags.get("penalty"))
        # both handles evaluate the penalty in float32 where it applies (the "float32" mode of PENALTY_MODES)
        replay_on_step_kernel(other, col, T, lambda r1, r2: rewards_agree(r1, r2, penalty, "float32"))
    else:
        other = r.twin(ROBOY_B200_GENERIC_FASTDIV="0")
        assert other.msj_kernels and not other.fast_division
        replay_on_step_kernel(other, col, T, bitwise)
    same_env_state(other, client)
    other.close()
    return r, m, sel


# ------------------------------------------------------------------------------------------------------------------- MSJ
@pytest.mark.parametrize("mode,ept", [("fp32", 1), ("tc", 1), ("tc_exact", 0)])
@pytest.mark.parametrize("flags", K1_FLAGS, ids=FLAG_IDS)
def test_msj_env_flags_in_the_fused_rollouts(flags, mode, ept):
    """n = 6001 is not a multiple of 4: the unaligned observation stores."""
    run_case("msj", flags, mode, ept)


@pytest.mark.parametrize("mode,ept,n", [("fp32", 2, 6001), ("tc", 2, 6001), ("tc", 3, 6001), ("fp32", 0, 40_017),
                                        ("tc", 0, 80_017)])
def test_kernel_variants_with_penalty_no_bonus_and_manual_reset(mode, ept, n):
    _, m, sel = run_case("msj", K1_FLAGS[-1], mode, ept, n)
    if n > 40_000:
        assert (mode == "fp32" and sel == 2) or (mode != "fp32" and m >= 2 * 8)   # E = 2, or groups walk several chunks


# ----------------------------------------------------------------------------------- MSJ-shaped robots with other limits
OTHER_FLAGS = [dict(), dict(penalty=True), dict(auto_reset=False)]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("flags", OTHER_FLAGS, ids=["default", "penalty", "manual_reset"])
@pytest.mark.parametrize("name", sorted(MSJ_SHAPED_OTHER_LIMITS))
def test_msj_shaped_robot_with_other_limits_in_the_fused_rollouts(name, flags, mode):
    """symmetric: hold centre 0, float32 penalty; one_sided: hold centre -1; asymmetric: hold action 0.5, asymmetric
    velocity space (no float32 penalty), and global env ids starting at 12,345 in its default-flag cases."""
    run_case(name, flags, mode, env_id_base=12_345 if (name, flags) == ("asymmetric", {}) else 0)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", sorted(ROBOTS))
def test_nan_weight_trips_the_action_error_on_every_robot(name, mode):
    r, _, _ = run_case(name, {}, mode, n=2001, nan=True)
    flags, first = r.client.errors()
    assert flags & orc.ERR_ACTION and first == 0
    assert torch.isnan(r.col.actions[:, :, 5]).all()


# ----------------------------------------------------------------------------------------- float32 vs float64 penalty
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", ["msj", "symmetric"])
def test_float32_penalty_keeps_every_exact_output_of_the_fused_rollouts(name, mode):
    """The penalty handle against one created under ROBOY_B200_PENALTY_F64=1: the same policy, so the same actions and
    the same exact outputs; rewards within PENALTY_REL, and more than n of them differ (the float32 chain ran)."""
    n = 6001
    h32, h64 = (Rollout(name, dict(penalty=True), mode, n=n, f64=f64) for f64 in (False, True))
    for h in (h32, h64):
        h.collect()
    a, b = h32.col, h64.col
    assert torch.equal(a.actions, b.actions) and torch.equal(a.obs, b.obs) and torch.equal(a.dones, b.dones)
    r32, r64 = a.rewards.double(), b.rewards.double()
    assert ((r32 - r64).abs() <= PENALTY_REL * r64.abs()).all()
    assert int((a.rewards != b.rewards).sum()) > n
    same_env_state(h32.client, h64.client)
    if name == "msj":
        assert h32.client.errors()[0] & orc.ERR_REWARD_RANGE   # the Stub's velocities break MSJ's reward_range


@pytest.mark.parametrize("name,mode", [("msj", m) for m in MODES] + [("symmetric", "tc_exact")])
def test_reward_range_bound_between_the_float32_and_the_float64_reward_in_the_fused_rollouts(name, mode):
    """reward_range[0] placed between the float32- and the float64-evaluated reward of env k at step t: inside the band
    the float64 expression decides, so the float32 handle counts the violations of the float64 handle, names the same
    first offender, and writes the float64 reward for that env."""
    hs = [Rollout(name, dict(penalty=True), mode, f64=f64) for f64 in (False, True)]
    for h in hs:
        h.collect()
    r32, r64 = (h.col.rewards.cpu().numpy() for h in hs)
    cand = np.argwhere((r32 != r64) & np.isfinite(r32) & np.isfinite(r64))
    assert len(cand) > hs[0].n
    cand = cand[np.argsort(r64[tuple(cand.T)])]
    for t, k in cand[[len(cand) // 4, len(cand) // 2, -len(cand) // 4]]:
        lo = (float(r32[t, k]) + float(r64[t, k])) / 2.0   # exact in float64; strictly between the two float32 rewards
        got = []
        for h in hs:
            h.restore()
            with environ(ROBOY_B200_PENALTY_F64="1" if h.f64 else "0"):
                h.client.set_reward_range(lo, float("inf"))
            assert h.client.penalty_float32 == (not h.f64)
            h.collect()
            got.append((float(h.col.rewards[t, k]), h.client.stats()["violations"], h.client.errors()))
        assert got[0][0] == got[1][0] == r64[t, k], (t, k, got)
        assert got[0][1:] == got[1][1:], (t, k, lo, got)
        assert got[0][1] > 0 and got[0][2][0] & orc.ERR_REWARD_RANGE
