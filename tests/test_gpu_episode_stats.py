"""The episode statistics (the 8-double vector ROBOY_STAT_* of every handle) of every producer against the CPU oracle.

Each producer reduces the vector its own way: K1 step_kernel, K1b rollout_kernel, the fused policy rollouts (float32 and
tensor-core), the generic step kernel and the external-simulator feed.  Per launch, the seven count fields and
sum_episode_len must equal the oracle's delta exactly (integers below 2^53).  sum_reward is checked against S64, the float64
sum of the rewards the kernel itself wrote (which are compared with the oracle elementwise at 1e-6): the kernels keep one
float32 partial per thread and add across threads in double, so a correct launch in which no thread adds more than m
rewards is within (m - 1) 2^-24 sum|r| + 1e-12 sum|r| of S64.  Where that bound is below half the smallest |r| of the
launch, one dropped, duplicated or dead-lane reward fails.
"""
import ctypes
import math

import numpy as np
import pytest
import torch

from cuda_adaptor import robot_from_bounds
from oracle import oracle as orc
from test_gpu_generic_robots import MSJ_SHAPED_OTHER_LIMITS, environ
from test_oracle_vs_reference import GENERIC_ROBOTS

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
RTOL = 1e-6
U32 = 2.0 ** -24
NAMES = orc.STAT_NAMES
I_REWARD = NAMES.index("sum_reward")
CAP = orc.STEP_MASK   # the step counter saturates here, next to the two held-state flag bits
ONE_JOINT = dict(dim_joint=1, dim_action=5, angle_low=-1.5, angle_high=2.0, vel_low=-0.4, vel_high=0.4, act_low=-0.3,
                 act_high=0.3)


def vec(d):
    return np.array([d[k] for k in NAMES], np.float64)


def check_delta(d, od, rewards, m, carried=0.0):
    """One launch: `d` the handle's stats delta, `od` the oracle's, `rewards` every reward the launch wrote, `m` an upper
    bound on the rewards one thread adds.  `carried`: |sum_reward| before the launch (the running total rounds each CTA's
    addition to its own ulp).  Returns (bound on |sum_reward - S64|, min |r|)."""
    for i, k in enumerate(NAMES):
        if i != I_REWARD:
            assert d[i] == od[i], (k, d[i], od[i])
    r = np.asarray(rewards.cpu().numpy() if torch.is_tensor(rewards) else rewards, np.float64).ravel()
    assert np.isfinite(r).all()
    s64, a = math.fsum(r), float(np.abs(r).sum())
    bound = (m - 1) * U32 * a + 1e-12 * (a + carried)
    assert abs(d[I_REWARD] - s64) <= bound, ("sum_reward", d[I_REWARD], s64, bound, m)
    return bound, float(np.abs(r).min())


class Tally:
    """Statistics of a handle and of its oracle, snapshotted so that each launch is checked on its own delta."""

    def __init__(self, client, ora):
        self.client, self.ora = client, ora
        self.g, self.o = vec(client.stats()), vec(ora.stats())

    def check(self, rewards, m, tight=False):
        g, o = vec(self.client.stats()), vec(self.ora.stats())
        bound, rmin = check_delta(g - self.g, o - self.o, rewards, m, abs(self.g[I_REWARD]))
        if tight:
            assert bound < 0.5 * rmin, ("bound not below half the smallest reward", bound, rmin, m)
        self.g, self.o = g, o


def make(n, seed, bounds=None, penalty=False, bonus=True, auto_reset=True, env_id_base=0):
    from gym_roboy_b200.envs import RoboyEnv
    from gym_roboy_b200.envs.simulations import CudaSimulationClient
    client = CudaSimulationClient(robot=robot_from_bounds(bounds), num_envs=n, seed=seed, env_id_base=env_id_base, device=DEV)
    env = RoboyEnv(client, joint_vel_penalty=penalty, is_agent_getting_bonus_for_reaching_goal=bonus, auto_reset=auto_reset,
                   strict=False)
    env._single = False
    ora = orc.OracleEnv(n, seed=seed, env_id_base=env_id_base, joint_vel_penalty=penalty, bonus=bonus, auto_reset=auto_reset,
                        threads=8, **(bounds or {}))
    env.reset(); ora.reset()
    return env, client, ora


def cdiv(a, b):
    return -(-a // b)


def m_step(client, T=1):
    """Rewards per thread of the step kernels (tuned K1 / K1b and generic): chunks of 32 envs per warp, times T."""
    g = client.step_geometry()
    return cdiv(cdiv(client.num_envs, 32), g["grid"] * g["block"] // 32) * T


def ragged_size(bounds=None):
    """2 x (threads of the capped step grid) + 17: some warp walks two chunks and more, and a ragged tail exists."""
    from gym_roboy_b200.envs.simulations import CudaSimulationClient
    probe = CudaSimulationClient(robot=robot_from_bounds(bounds), num_envs=1 << 21, seed=0, device=DEV)
    g = probe.step_geometry()
    probe.close()
    n = 2 * g["grid"] * g["block"] + 17
    assert n < 1 << 21
    return n


def set_phases(client, ora, steps, idx=None):
    steps = np.asarray(steps, np.int64)
    client.set_step_num(steps.astype(np.int32), idx=idx)
    sl = slice(None) if idx is None else idx
    ora.step_flags[sl] = (ora.step_flags[sl] & ~np.uint32(CAP)) | steps.astype(np.uint32)


def inject_held(client, ora, rng, idx, feasible):
    """float32 held states (some with velocities far outside the velocity space: with the penalty their reward leaves
    reward_range) on envs `idx`; `feasible` False sets the held-infeasible flag bit."""
    J = ora.J
    lo, hi = ora.bounds["angle_low"], ora.bounds["angle_high"]
    q = rng.uniform(lo, hi, (idx.size, J)).astype(np.float32)
    qd = rng.uniform(-0.3, 0.3, (idx.size, J)).astype(np.float32)
    qd[::3] = np.float32(10.0)
    client.set_state(q, qd, feasible.astype(np.uint8), idx=idx)
    ora.held[:J, idx] = q.T
    ora.held[J:, idx] = qd.T
    ora.step_flags[idx] = (ora.step_flags[idx] & np.uint32(CAP)) | np.where(feasible, 0, orc.F_HELD_INFEASIBLE).astype(np.uint32)


def populate(client, ora, rng):
    """Phases spread over 1..400 and a held state on 2 % of the envs (half of them infeasible).  Returns those envs."""
    n = client.num_envs
    set_phases(client, ora, rng.integers(1, 401, n))
    held = np.sort(rng.choice(n, max(n // 50, 1), replace=False))
    inject_held(client, ora, rng, held, rng.random(held.size) < 0.5)
    return held


def plant_goals(client, ora, rng, seed):
    """Goals at the threshold distance (x (1 -+ 1e-7), 0.7, 1.2) from the state the next step samples: successes."""
    J, n = ora.J, ora.n
    lo, hi = ora.bounds["angle_low"], ora.bounds["angle_high"]
    gids = np.arange(n, dtype=np.uint64) + np.uint64(ora.cfg.env_id_base)
    q, _ = orc.draw_state(seed, gids, ora.counter + 1, lo, hi, J=J)
    thr_a, _ = orc.thresholds(ora.cfg)
    d = rng.normal(size=(n, J)); d /= np.linalg.norm(d, axis=1, keepdims=True)
    r = float(thr_a) * (1 + rng.choice([-1e-7, 1e-7, -0.3, 0.2], n))
    g = np.clip(q.astype(np.float64) + d * r[:, None], lo, hi).astype(np.float32)
    client.set_goal(g); ora.goal[:] = g.T


def actions(rng, ora, held=None, hold_frac=0.02):
    """Uniform actions with hold rows, the injected held states through the hold branch, out-of-range and NaN rows."""
    n, A = ora.n, ora.A
    hold_act, _ = orc.hold_action(ora.bounds)
    a = rng.uniform(-1, 1, (n, A)).astype(np.float32)
    a[rng.random(n) < hold_frac] = hold_act
    if held is not None:
        a[held[::2]] = hold_act
    a[rng.random(n) < 0.002] = np.float32(1.5)
    nan_rows = np.flatnonzero(rng.random(n) < 0.002)
    a[nan_rows, rng.integers(0, A, nan_rows.size)] = np.nan
    return a


def check_outputs(obs, rew, done, o, r, d, t=None):
    obs, rew, done = (x.cpu().numpy() if torch.is_tensor(x) else np.asarray(x) for x in (obs, rew, done))
    assert np.array_equal(done.astype(bool), d), ("done", t)
    assert np.array_equal(obs, o), ("obs", t)
    rel = np.abs(rew.astype(np.float64) - r) / np.maximum(np.abs(r.astype(np.float64)), 1e-30)
    assert rel.max() <= RTOL, ("reward", t, rel.max())


def check_state(client, ora):
    assert np.array_equal(client.goal.cpu().numpy(), ora.goal)
    assert np.array_equal(client.step_flags.cpu().numpy().view(np.uint32), ora.step_flags)


def fused_steps(client, ora, rng, seed, steps, m, held=None, tight=False):
    tally = Tally(client, ora)
    for t in range(steps):
        if t % 2 == 0:
            plant_goals(client, ora, rng, seed)
        a = actions(rng, ora, held)
        client.step_fused(torch.as_tensor(a, device=DEV))
        o, r, d = ora.step(a)
        check_outputs(client.obs, client.reward, client.done_u8, o, r, d, t)
        tally.check(client.reward, m, tight)
    check_state(client, ora)
    return vec(client.stats())


# ------------------------------------------------------------------------------------------------------------ K1 step_kernel
K1_FLAGS = [dict(), dict(penalty=True), dict(bonus=False), dict(auto_reset=False),
            dict(penalty=True, bonus=False, auto_reset=False)]


@pytest.mark.parametrize("flags", K1_FLAGS, ids=["default", "penalty", "nobonus", "manual_reset", "penalty_nobonus_manual"])
def test_step_kernel_statistics(flags):
    n, seed = ragged_size(), 1234
    _, client, ora = make(n, seed, **flags)
    assert client.msj_kernels and client.fast_division
    rng = np.random.default_rng(1)
    held = populate(client, ora, rng)
    m = m_step(client)
    assert m >= 3
    s = fused_steps(client, ora, rng, seed, 3, m, held, tight=not flags.get("penalty"))
    so = vec(ora.stats())
    assert all(s[NAMES.index(k)] > 0 for k in ("episodes", "successes", "timeouts", "holds", "violations")), s
    if flags.get("penalty"):
        assert ora.errors()[0] & orc.ERR_REWARD_RANGE
    assert s[NAMES.index("sum_episode_len")] == so[NAMES.index("sum_episode_len")]


@pytest.mark.parametrize("ieee", [False, True], ids=["checked_division", "ieee_division"])
def test_step_kernel_statistics_of_an_msj_shaped_robot_with_other_limits(ieee):
    b = MSJ_SHAPED_OTHER_LIMITS["asymmetric"]
    n, seed = ragged_size(b), 17
    with environ(**({"ROBOY_B200_GENERIC_FASTDIV": "0"} if ieee else {})):
        _, client, ora = make(n, seed, b)
    assert client.msj_kernels and client.fast_division != ieee
    rng = np.random.default_rng(2)
    held = populate(client, ora, rng)
    fused_steps(client, ora, rng, seed, 3, m_step(client), held, tight=True)


# --------------------------------------------------------------------------------------------------- K1b rollout_kernel
@pytest.mark.parametrize("T", [1, 5, 64])
@pytest.mark.parametrize("auto_reset", [True, False])
def test_open_loop_statistics(T, auto_reset):
    n, seed = (ragged_size() if T < 64 else 20_033), 31
    _, client, ora = make(n, seed, penalty=not auto_reset, auto_reset=auto_reset)
    rng = np.random.default_rng(T)
    held = populate(client, ora, rng)
    set_phases(client, ora, 400 - (np.arange(n) % (T + 2)))   # episode ends inside the window
    plant_goals(client, ora, rng, seed)
    acts = np.stack([actions(rng, ora, held) for _ in range(T)])
    tally = Tally(client, ora)
    obs, rew, done = client.step_many(torch.as_tensor(acts, device=DEV))
    for t in range(T):
        o, r, d = ora.step(acts[t])
        check_outputs(obs[t], rew[t], done[t], o, r, d, t)
    m = m_step(client, T)
    tally.check(rew, m, tight=T == 1 and auto_reset)
    check_state(client, ora)
    assert ora.stats()["episodes"] >= n // 3


# ------------------------------------------------------------------------------------------------------------- host path
@pytest.mark.parametrize("mode,n_streams", [("staged", 1), ("staged", 2), ("mapped_out", 2), ("mapped_all", 2)])
def test_host_path_statistics(mode, n_streams):
    from gym_roboy_b200 import _native
    n, seed = 30_011, 8   # stages of 4,096 do not divide n
    _, client, ora = make(n, seed, penalty=True)
    client.set_host_pipeline(stage_envs=4096, n_streams=n_streams)
    client.set_host_mode({"staged": _native.HOST_STAGED, "mapped_out": _native.HOST_MAPPED_OUT,
                          "mapped_all": _native.HOST_MAPPED_ALL}[mode])
    rng = np.random.default_rng(4)
    held = populate(client, ora, rng)
    a_h, obs_h, rew_h, done_h = client.host_buffers()
    tally = Tally(client, ora)
    m = m_step(client)   # a stage's grid walks at most as many chunks per warp as the whole population's
    for t in range(3):
        plant_goals(client, ora, rng, seed)
        a_h[...] = actions(rng, ora, held)
        client.step_host(a_h, obs_h, rew_h, done_h)
        o, r, d = ora.step(np.array(a_h))
        check_outputs(obs_h, rew_h, done_h, o, r, d, t)
        tally.check(np.array(rew_h), m, tight=True)
    check_state(client, ora)


# ------------------------------------------------------------------------------------------- K5 / K6 fused policy rollouts
def policy_m(client, mode, ept, T):
    """Rewards per thread of the fused policy rollout launch, from the geometry the library reports."""
    from gym_roboy_b200 import _native
    lib, n = _native.load(), client.num_envs
    grid, block, smem, sel = ctypes.c_int(), ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    if mode == "fp32":
        _native.check(lib.roboy_policy_geometry(client._h, ept, ctypes.byref(grid), ctypes.byref(block), ctypes.byref(smem),
                                                ctypes.byref(sel)))
        E = sel.value
        return cdiv(cdiv(n, 32 * E), grid.value * block.value // 32) * T * E, E, grid.value
    _native.check(lib.roboy_policy_tc_geometry(client._h, ept, int(mode == "tc_exact"), ctypes.byref(grid), ctypes.byref(block),
                                               ctypes.byref(smem), ctypes.byref(sel)))
    tiles = 2 if sel.value == 2 else 1   # variant 2: two 128-env tiles per group of 128 threads
    return cdiv(cdiv(n, 128 * tiles), grid.value * block.value // 128) * T * tiles, sel.value, grid.value


def make_rollout(n, seed, T, mode, ept, auto_reset=True):
    from gym_roboy_b200.rollout import MlpPolicy, RolloutCollector
    env, client, ora = make(n, seed, auto_reset=auto_reset)
    torch.manual_seed(0)
    policy = MlpPolicy().to(DEV)
    with torch.no_grad():
        policy.log_std.copy_(torch.linspace(-1.0, 0.7, 8))   # a few actions beyond [-1, 1]: clipped
    col = RolloutCollector(env, policy, n_steps=T, fused=mode, noise_seed=5, envs_per_thread=ept)
    ora.reset()
    return client, ora, col


def replay_rollout(client, ora, col, T):
    acts = np.clip(col.actions.cpu().numpy(), -1.0, 1.0)
    obs, rew, done = col.obs.cpu().numpy(), col.rewards.cpu().numpy(), col.dones.cpu().numpy()
    for t in range(T):
        o, r, d = ora.step(acts[t])
        check_outputs(obs[t + 1] if t + 1 < T else col.obs[T].cpu().numpy(), rew[t], done[t], o, r, d, t)


@pytest.mark.parametrize("mode,ept,n", [("fp32", 1, 6001), ("fp32", 2, 6001), ("fp32", 0, 40_017), ("tc", 1, 6001),
                                        ("tc", 2, 6001), ("tc", 3, 6001), ("tc", 0, 80_017), ("tc_exact", 0, 6001),
                                        ("tc_exact", 0, 80_017)])
def test_policy_rollout_statistics(mode, ept, n):
    T, seed = 4, 21
    client, ora, col = make_rollout(n, seed, T, mode, ept)
    rng = np.random.default_rng(5)
    set_phases(client, ora, rng.integers(380, 401, n))
    m, sel, _ = policy_m(client, mode, ept, T)
    if n > 40_000:
        assert (mode == "fp32" and sel == 2) or (mode != "fp32" and m >= 2 * T)   # E = 2, or groups walk several chunks
    tally = Tally(client, ora)
    col.collect()
    torch.cuda.synchronize()
    replay_rollout(client, ora, col, T)
    tally.check(col.rewards, m, tight=n < 10_000)
    check_state(client, ora)
    s = ora.stats()
    assert s["episodes"] > 0 and s["violations"] == 0


def test_policy_rollout_holds_and_nan_actions_are_counted():
    n, T = 3001, 3
    for mode in ("fp32", "tc", "tc_exact"):
        client, ora, col = make_rollout(n, 9, T, mode, 0)
        set_phases(client, ora, np.arange(n) % 400 + 1)
        m, _, _ = policy_m(client, mode, 0, T)
        tally = Tally(client, ora)
        with torch.no_grad():
            for p_ in col.policy.pi.parameters():
                p_.zero_()
            col.policy.log_std.fill_(-40.0)                     # actions ~ 0: the hold branch
        for what in ("holds", "violations"):
            if what == "violations":
                with torch.no_grad():
                    col.policy.pi[4].bias[5] = float("nan")     # every action NaN in one component
            before = ora.stats()[what]
            col.collect()
            torch.cuda.synchronize()
            replay_rollout(client, ora, col, T)
            tally.check(col.rewards, m, tight=True)
            assert ora.stats()[what] - before == n * T, (mode, what)


# ---------------------------------------------------------------------------------------------------- generic step kernel
GENERIC_CASES = {"one_joint": ONE_JOINT, "six_joints_14_tendons": GENERIC_ROBOTS["six_joints_14_tendons"],
                 "fifteen_joints_64_tendons": GENERIC_ROBOTS["fifteen_joints_64_tendons"]}


@pytest.mark.parametrize("penalty", [False, True])
@pytest.mark.parametrize("name", sorted(GENERIC_CASES))
def test_generic_step_statistics(name, penalty):
    b = GENERIC_CASES[name]
    n, seed = (ragged_size(b) if name != "fifteen_joints_64_tendons" else 40_009), 6
    _, client, ora = make(n, seed, b, penalty=penalty)
    assert not client.msj_kernels
    rng = np.random.default_rng(6)
    held = populate(client, ora, rng)
    m = m_step(client)
    # (the one-joint robot reaches its planted goals often: its bonus rewards make sum|r| too large for a tight bound)
    fused_steps(client, ora, rng, seed, 3, m, held, tight=m == 1 or (name, penalty) == ("six_joints_14_tendons", False))
    s = ora.stats()
    assert s["episodes"] > 0 and s["violations"] > 0


def test_msj_on_the_generic_kernel_counts_what_the_tuned_kernel_counts():
    n, seed, T = ragged_size(), 3, 3
    _, tuned, ora = make(n, seed, penalty=True)
    with environ(ROBOY_B200_FORCE_GENERIC="1"):
        _, gen, _ = make(n, seed, penalty=True)
    assert tuned.msj_kernels and not gen.msj_kernels
    rng = np.random.default_rng(7)
    held = populate(tuned, ora, rng)
    rng2 = np.random.default_rng(7)
    populate(gen, orc.OracleEnv(n, seed=seed, joint_vel_penalty=True), rng2)
    for t in range(T):
        a = torch.as_tensor(actions(rng, ora, held), device=DEV)
        g0, t0 = vec(gen.stats()), vec(tuned.stats())
        gen.step_fused(a)
        tuned.step_fused(a)
        dg, dt = vec(gen.stats()) - g0, vec(tuned.stats()) - t0
        check_delta(dg, dt, gen.reward, m_step(gen))   # count fields identical
        check_delta(dt, dg, tuned.reward, m_step(tuned))
        assert torch.equal(gen.done_u8, tuned.done_u8)
    assert vec(tuned.stats())[NAMES.index("episodes")] > 0


# ------------------------------------------------------------------------------------------------------- external feed
def test_external_feed_statistics():
    n, seed = 20_011, 12
    _, client, ora = make(n, seed, penalty=True)
    rng = np.random.default_rng(8)
    set_phases(client, ora, rng.integers(1, 401, n))
    tally = Tally(client, ora)
    for t in range(4):
        q = rng.uniform(-3.2, 3.2, (n, 3)).astype(np.float32)        # some outside the angle space
        goal = client.goal.cpu().numpy().T
        near = rng.random(n) < 0.3
        q[near] = goal[near] + np.float32(1e-3)                      # successes
        qd = rng.uniform(-0.6, 0.6, (n, 3)).astype(np.float32)
        qd[near] = 0.0
        feas = (rng.random(n) < 0.8).astype(np.uint8)
        client.step_external(q, qd, feas)
        o, r, d = ora.step_external(q, qd, feas)
        check_outputs(client.obs, client.reward, client.done_u8, o, r, d, t)
        tally.check(client.reward, 1, tight=True)
    s = ora.stats()
    assert s["successes"] > 0 and s["timeouts"] > 0 and s["violations"] > 0
    check_state(client, ora)


# ------------------------------------------------------------------------------------------------------------ invariants
def test_clear_stats_and_the_dlpack_view():
    n = 5000
    _, client, ora = make(n, 2)
    rng = np.random.default_rng(9)
    held = populate(client, ora, rng)
    for _ in range(3):
        client.step_fused(torch.as_tensor(actions(rng, ora, held), device=DEV))
        assert np.array_equal(client.stats_tensor.cpu().numpy(), vec(client.stats()))
    assert vec(client.stats())[NAMES.index("violations")] > 0
    client.clear_stats()
    assert not vec(client.stats()).any() and not client.stats_tensor.any()
    assert client.errors() == (0, None)


def test_resumed_handle_continues_the_totals():
    n, seed = 40_003, 4
    env, client, ora = make(n, seed, penalty=True)
    rng = np.random.default_rng(10)
    held = populate(client, ora, rng)
    acts = [torch.as_tensor(actions(rng, ora, held), device=DEV) for _ in range(8)]
    for a in acts[:4]:
        client.step_fused(a)
    client.clear_errors()
    sd = client.state_dict()
    for a in acts[4:]:
        client.step_fused(a)
    whole = vec(client.stats())
    _, client2, _ = make(n, 999, penalty=True)
    client2.load_state_dict(sd)
    for a in acts[4:]:
        client2.step_fused(a)
    resumed = vec(client2.stats())
    for i, k in enumerate(NAMES):
        if i == I_REWARD:
            assert abs(resumed[i] - whole[i]) <= 1e-12 * abs(whole[i]), k
        else:
            assert resumed[i] == whole[i], k


def test_done_index_and_terminal_observations_leave_the_statistics_alone():
    n, seed = 30_001, 7
    _, plain, ora = make(n, seed)
    _, side, _ = make(n, seed)
    side.enable_done_index(True)
    side.enable_terminal_obs(True)
    rng = np.random.default_rng(11)
    steps = rng.integers(1, 401, n).astype(np.int32)
    plain.set_step_num(steps); side.set_step_num(steps)
    for _ in range(5):
        a = torch.as_tensor(actions(rng, ora), device=DEV)
        plain.step_fused(a)
        side.step_fused(a)
        side.done_indices(with_terminal_obs=True)
        s1, s2 = vec(plain.stats()), vec(side.stats())
        assert np.array_equal(np.delete(s1, I_REWARD), np.delete(s2, I_REWARD))
        assert abs(s1[I_REWARD] - s2[I_REWARD]) <= 1e-12 * abs(s1[I_REWARD])
    assert vec(plain.stats())[NAMES.index("episodes")] > 0


def test_two_half_shards_count_what_the_full_shard_counts():
    n, seed, T = 20_000, 77, 6
    rng = np.random.default_rng(12)
    ora_full = orc.OracleEnv(n, seed=seed)
    acts = [actions(rng, ora_full) for _ in range(T)]
    steps = rng.integers(1, 401, n).astype(np.int32)
    totals = []
    for shards in ([(0, n)], [(0, n // 2), (n // 2, n)]):
        tot = np.zeros(len(NAMES))
        for b, e in shards:
            _, client, _ = make(e - b, seed, env_id_base=b)
            client.set_step_num(steps[b:e])
            for a in acts:
                client.step_fused(torch.as_tensor(a[b:e], device=DEV))
            tot += vec(client.stats())
        totals.append(tot)
    assert np.array_equal(np.delete(totals[0], I_REWARD), np.delete(totals[1], I_REWARD))
    assert totals[0][NAMES.index("episodes")] > 0


# ------------------------------------------------------------------------------------------------ the step-counter cap
def at_the_cap(client, ora, rng):
    """Step counters at 2^24 - 2 and 2^24 - 1; a third of the envs carry the held-infeasible flag, a third a feasible
    float32 held state, the rest the zero-state flag a reset leaves."""
    n = client.num_envs
    set_phases(client, ora, np.where(np.arange(n) % 2 == 0, CAP - 1, CAP))
    part = np.arange(n) % 3
    for k, feas in ((0, False), (1, True)):
        idx = np.flatnonzero(part == k)
        inject_held(client, ora, rng, idx, np.full(idx.size, feas))
    flags = ora.step_flags & ~np.uint32(CAP)
    assert (flags == orc.F_HELD_INFEASIBLE).any() and (flags == orc.F_HELD_ZERO64).any()


CAP_FLAGS = [True, False]


@pytest.mark.parametrize("auto_reset", CAP_FLAGS)
def test_step_counter_cap_step_kernel(auto_reset):
    n, seed = ragged_size(), 41
    _, client, ora = make(n, seed, auto_reset=auto_reset)
    rng = np.random.default_rng(13)
    at_the_cap(client, ora, rng)
    assert n // client.step_geometry()["grid"] > 256   # one CTA's episode lengths pass 2^32 in the first launch
    tally = Tally(client, ora)
    for t in range(2):
        a = actions(rng, ora, hold_frac=0.3)
        client.step_fused(torch.as_tensor(a, device=DEV))
        o, r, d = ora.step(a)
        check_outputs(client.obs, client.reward, client.done_u8, o, r, d, t)
        tally.check(client.reward, m_step(client))
        check_state(client, ora)
    assert ora.stats()["sum_episode_len"] >= n * (CAP - 1)


@pytest.mark.parametrize("auto_reset", CAP_FLAGS)
def test_step_counter_cap_open_loop(auto_reset):
    n, seed, T = ragged_size(), 42, 3
    _, client, ora = make(n, seed, auto_reset=auto_reset)
    rng = np.random.default_rng(14)
    at_the_cap(client, ora, rng)
    acts = np.stack([actions(rng, ora, hold_frac=0.3) for _ in range(T)])
    tally = Tally(client, ora)
    obs, rew, done = client.step_many(torch.as_tensor(acts, device=DEV))
    for t in range(T):
        o, r, d = ora.step(acts[t])
        check_outputs(obs[t], rew[t], done[t], o, r, d, t)
    assert (n // client.step_geometry()["grid"]) * (1 if auto_reset else T) > 256
    tally.check(rew, m_step(client, T))
    check_state(client, ora)


@pytest.mark.parametrize("mode,n", [("fp32", 40_017), ("tc", 80_017), ("tc_exact", 80_017)])
@pytest.mark.parametrize("auto_reset", CAP_FLAGS)
def test_step_counter_cap_policy_rollout(mode, n, auto_reset):
    T = 3
    client, ora, col = make_rollout(n, 43, T, mode, 0, auto_reset=auto_reset)
    rng = np.random.default_rng(15)
    at_the_cap(client, ora, rng)
    m, _, grid = policy_m(client, mode, 0, T)
    assert (n // grid) * (1 if auto_reset else T) > 256   # one CTA's episode lengths pass 2^32
    tally = Tally(client, ora)
    col.collect()
    torch.cuda.synchronize()
    replay_rollout(client, ora, col, T)
    tally.check(col.rewards, m)
    check_state(client, ora)


@pytest.mark.parametrize("auto_reset", CAP_FLAGS)
def test_step_counter_cap_generic_external_and_host(auto_reset):
    b = GENERIC_ROBOTS["six_joints_14_tendons"]
    n, seed = 20_011, 44
    # generic step kernel
    _, client, ora = make(n, seed, b, auto_reset=auto_reset)
    rng = np.random.default_rng(16)
    at_the_cap(client, ora, rng)
    tally = Tally(client, ora)
    for t in range(2):
        a = actions(rng, ora, hold_frac=0.3)
        client.step_fused(torch.as_tensor(a, device=DEV))
        o, r, d = ora.step(a)
        check_outputs(client.obs, client.reward, client.done_u8, o, r, d, t)
        tally.check(client.reward, m_step(client))
        check_state(client, ora)
    # external feed
    _, client, ora = make(n, seed, auto_reset=auto_reset)
    at_the_cap(client, ora, rng)
    tally = Tally(client, ora)
    for t in range(2):
        q = rng.uniform(-3.0, 3.0, (n, 3)).astype(np.float32)
        qd = rng.uniform(-0.5, 0.5, (n, 3)).astype(np.float32)
        client.step_external(q, qd)
        o, r, d = ora.step_external(q, qd)
        check_outputs(client.obs, client.reward, client.done_u8, o, r, d, t)
        tally.check(client.reward, 1)
        check_state(client, ora)
    # host path (stages of the tuned step kernel)
    n = ragged_size()
    _, client, ora = make(n, seed, auto_reset=auto_reset)
    client.set_host_pipeline(stage_envs=1 << 17, n_streams=2, ramp=False)
    assert (1 << 17) < n and (1 << 17) // client.step_geometry()["grid"] > 256   # the first stage's CTAs pass 2^32
    at_the_cap(client, ora, rng)
    a_h, obs_h, rew_h, done_h = client.host_buffers()
    tally = Tally(client, ora)
    for t in range(2):
        a_h[...] = actions(rng, ora, hold_frac=0.3)
        client.step_host(a_h, obs_h, rew_h, done_h)
        o, r, d = ora.step(np.array(a_h))
        check_outputs(obs_h, rew_h, done_h, o, r, d, t)
        tally.check(np.array(rew_h), m_step(client))
        check_state(client, ora)
