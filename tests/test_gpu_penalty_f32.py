"""The velocity penalty of roboy_env.py:98-100 on the sampled-state path, float32 with a float64 re-run near the bounds of
reward_range (PenaltyF32, gym_roboy_b200/csrc/msj_math.cuh) against a handle kept on the float64 expression
(ROBOY_B200_PENALTY_F64=1): every bit-exact output stays bit-exact -- observations, done mask, goals, step words, the
error word of the reward_range assert (:109), its first offending env and the violation count -- and the rewards agree far
inside north_star's 1e-6."""
import os

import numpy as np
import pytest
import torch

from cuda_adaptor import robot_from_bounds
from oracle import oracle as orc
from test_oracle_vs_reference import GENERIC_ROBOTS

pytestmark = pytest.mark.gpu
REL = 5e-7   # (J/2 + 4) roundings of 2^-24 at J <= 8 (msj_math.cuh): at most 4.8e-7
ROBOTS = {   # symmetric velocity spaces, at most 8 joints: where the float32 evaluation applies
    "msj": {},
    "six_joints_14_tendons": GENERIC_ROBOTS["six_joints_14_tendons"],                  # generic kernels
    "msj_shaped_other_limits": dict(angle_low=-2.0, angle_high=2.0, vel_low=-0.7, vel_high=0.7, act_low=-0.1, act_high=0.4),
    "five_joints_per_component": dict(angle_low=[-3.1, -1.0, -2.0, -0.7, -1.3], angle_high=[3.1, 1.0, 2.5, 0.9, 1.3],
                                      vel_low=[-0.5, -0.4, -0.3, -0.2, -0.1], vel_high=[0.5, 0.4, 0.3, 0.2, 0.1],
                                      dim_action=11, act_low=-0.25, act_high=0.25),
}


def make(robot, n, seed, bonus, f64):
    from gym_roboy_b200.envs import RoboyEnv
    from gym_roboy_b200.envs.simulations import CudaSimulationClient
    if f64:
        os.environ["ROBOY_B200_PENALTY_F64"] = "1"
    try:
        kw = {"robot": robot_from_bounds(robot)} if robot else {}
        client = CudaSimulationClient(num_envs=n, seed=seed, device="cuda:0", **kw)
        env = RoboyEnv(client, joint_vel_penalty=True, is_agent_getting_bonus_for_reaching_goal=bonus, strict=False)
        assert client.penalty_float32 == (not f64)
    finally:
        os.environ.pop("ROBOY_B200_PENALTY_F64", None)
    return env, client


def actions(rng, n, b):
    zero_action, can_hold = orc.hold_action(b)
    assert can_hold
    a = rng.uniform(-1, 1, (n, zero_action.size)).astype(np.float32)
    a[rng.random(n) < 0.03] = zero_action   # Stub holds (simulation_client.py:38): the general path, float64 in both handles
    return torch.as_tensor(a, device="cuda:0")


def rel_err(r32, r64):
    a, b = r32.double(), r64.double()
    return ((a - b).abs() / b.abs().clamp_min(1e-30)).max().item()


@pytest.mark.parametrize("bonus", [True, False])
@pytest.mark.parametrize("robot", sorted(ROBOTS))
def test_float32_penalty_keeps_every_exact_output(robot, bonus):
    b = ROBOTS[robot]
    n, T = 300_001, 24
    e32, c32 = make(b, n, 11, bonus, False)
    e64, c64 = make(b, n, 11, bonus, True)
    assert e32.reward_range == e64.reward_range
    assert torch.equal(e32.reset(), e64.reset())
    steps = (np.arange(n) % 400 + 1).astype(np.int32)
    c32.set_step_num(steps); c64.set_step_num(steps)
    rng = np.random.default_rng(5)
    differing, worst = 0, 0.0
    for t in range(T):
        a = actions(rng, n, b)
        o1, r1, d1, _ = e32.step(a)
        o2, r2, d2, _ = e64.step(a)
        assert torch.equal(o1, o2) and torch.equal(d1, d2), t
        worst = max(worst, rel_err(r1, r2))
        differing += int((r1 != r2).sum().item())
    assert worst <= REL, worst
    print("worst relative difference between the float32 and the float64 penalty: %.3g (%s)" % (worst, robot))
    assert differing > n, "the float32 path never ran"   # about half of all rewards round differently
    assert torch.equal(c32.goal, c64.goal) and torch.equal(c32.step_flags, c64.step_flags)
    assert c32.errors() == c64.errors()
    if robot == "msj":
        assert c32.errors()[0] & 2   # the Stub's velocities (drawn from the angle space) break MSJ's reward_range (DESIGN 2)
    s32, s64 = c32.stats(), c64.stats()
    for k in s32:
        if k == "sum_reward":
            assert abs(s32[k] - s64[k]) <= 1e-6 * abs(s64[k])
        else:
            assert s32[k] == s64[k], (k, s32[k], s64[k])
    assert s32["holds"] > 0 and s32["episodes"] > 0 and (s32["violations"] > 0 or robot != "msj")


@pytest.mark.parametrize("robot", ["msj", "six_joints_14_tendons"])
def test_reward_range_bound_between_the_float32_and_the_float64_reward(robot):
    """reward_range[0] placed BETWEEN an env's float32-evaluated and float64-evaluated reward: a float32 comparison would
    put that env on the wrong side of the assert; inside the band the float64 expression decides, so both handles count
    the same violations and name the same first offender."""
    b = ROBOTS[robot]
    n, seed = 200_003, 23
    rng = np.random.default_rng(9)
    e32, c32 = make(b, n, seed, True, False)
    e64, c64 = make(b, n, seed, True, True)
    a = actions(rng, n, b)
    e32.reset(); e64.reset()
    _, r1, _, _ = e32.step(a)
    _, r2, _, _ = e64.step(a)
    r1, r2 = r1.cpu().numpy(), r2.cpu().numpy()
    cand = np.flatnonzero((r1 != r2) & np.isfinite(r1) & np.isfinite(r2))
    assert cand.size > n // 10
    picks = list(cand[np.argsort(r2[cand])][[cand.size // 50, cand.size // 4, cand.size // 2, -cand.size // 4, -cand.size // 50]])
    for k in picks:
        lo = (float(r1[k]) + float(r2[k])) / 2.0   # exact in float64; strictly between the two float32 rewards
        counts, firsts, rewards = [], [], []
        for f64 in (False, True):
            env, client = make(b, n, seed, True, f64)
            # the library re-reads ROBOY_B200_PENALTY_F64 with a new reward range: keep the float64 handle on float64
            if f64:
                os.environ["ROBOY_B200_PENALTY_F64"] = "1"
            try:
                client.set_reward_range(lo, float("inf"))
            finally:
                os.environ.pop("ROBOY_B200_PENALTY_F64", None)
            assert client.penalty_float32 == (not f64)
            env.reset()
            _, r, _, _ = env.step(a)
            rewards.append(r.cpu().numpy())
            counts.append(client.stats()["violations"])
            firsts.append(client.errors())
        # the env itself took the float64 expression in the float32 handle: same bits there
        assert rewards[0][k] == rewards[1][k] == r2[k]
        assert counts[0] == counts[1] and firsts[0] == firsts[1], (k, lo, counts, firsts)
        # and the count is the float64 one: envs whose float64-evaluated reward lies below lo
        # (r2 is that reward rounded to float32; only env k can sit within half an ulp of lo)
        expect = int((np.delete(r2, k).astype(np.float64) < lo).sum())
        assert abs(counts[1] - expect) <= 3


def test_float32_penalty_is_off_where_its_error_bound_does_not_hold():
    from gym_roboy_b200.envs.simulations import CudaSimulationClient
    # more than 8 joints: the bound (J/2 + 3) * 2^-24 no longer leaves room below 1e-6
    c = CudaSimulationClient(robot=robot_from_bounds(GENERIC_ROBOTS["fifteen_joints_64_tendons"]), num_envs=64, seed=1, device="cuda:0")
    assert not c.penalty_float32
    # an asymmetric velocity space: the goal's normalised zero velocity is not a float32 value
    asym = dict(dim_joint=3, dim_action=8, angle_low=-1.0, angle_high=2.0, vel_low=-0.3, vel_high=1.0, act_low=0.0, act_high=0.3)
    c = CudaSimulationClient(robot=robot_from_bounds(asym), num_envs=64, seed=1, device="cuda:0")
    assert not c.penalty_float32
    assert CudaSimulationClient(num_envs=64, seed=1, device="cuda:0").penalty_float32
