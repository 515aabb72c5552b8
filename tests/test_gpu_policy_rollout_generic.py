"""The float32 fused policy rollout (`roboy_policy_rollout`) on robots other than MSJ: the generic kernel
(roboy_policy_generic.cu), one instantiation per joint count.

Each case prepares a population (step counters spread over 1..400 with a cluster at the timeout, injected held states,
some infeasible and some with velocities of 1000, goals planted on both sides of the reached threshold), runs ONE
rollout with its noise recorded, and checks:
  * the policy outputs against the torch float32 MlpPolicy(3J, A): values, mean + std * z, logp;
  * the noise against a numpy restatement of its definition (normal k: Philox block (stream 4, sub k // 4), word pair
    (k % 4) // 2, Box-Muller, first or second value by k % 2);
  * the env outputs against the CPU oracle on clip(actions): obs / done / goals / step words / error word and first
    offender exact, rewards to 1e-6, the statistics delta within the bound of test_gpu_episode_stats;
  * the env outputs against T calls of the generic step kernel on a second handle restored from the snapshot: bit for
    bit, rewards included.
MSJ forced onto the generic rollout is compared with the MSJ kernel (K5) on the same seeds: the same bits.
"""
import ctypes
import math

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from test_gpu_episode_stats import CAP, Tally, check_outputs, check_state, inject_held, make, policy_m, set_phases
from test_gpu_generic_robots import PENALTY_REL, environ, rewards_agree
from test_gpu_policy_rollout_envs import bitwise, errors_equal, plant_goals, replay_on_step_kernel, same_env_state
from test_oracle_vs_reference import GENERIC_ROBOTS, random_robot

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
TOL = dict(rtol=1e-5, atol=2e-5)   # the MSJ kernel's tolerances (test_gpu_policy_rollout.POLICY_TOL["fp32"])
NOISE_SEED = 5


def numpy_noise(noise_seed, gids, t, A):
    """Restatement of the rollout's noise for A actions: ceil(A / 4) Philox blocks (stream 4, sub 0, 1, ...), each two
    Box-Muller pairs; the normals past A of the last block are discarded."""
    z = []
    for sub in range((A + 3) // 4):
        x = orc._block(noise_seed, gids, t, 4, sub)
        for a, b in ((x[0], x[1]), (x[2], x[3])):
            u1 = (a >> np.uint32(8)).astype(np.float64) * 2.0 ** -24 + 2.0 ** -25
            u2 = (b >> np.uint32(8)).astype(np.float64) * 2.0 ** -24
            r = np.sqrt(-2.0 * np.log(u1))
            z += [r * np.cos(2 * np.pi * u2), r * np.sin(2 * np.pi * u2)]
    return np.stack(z[:A], axis=-1)


def hold_intervals(client):
    """Per tendon, the float32 interval of actions the Stub holds at (roboy_hold_intervals)."""
    from gym_roboy_b200 import _native
    lo, hi = (ctypes.c_float * 64)(), (ctypes.c_float * 64)()
    _native.check(_native.load().roboy_hold_intervals(ctypes.byref(client._cfg), lo, hi))
    A = client.dim_action
    return np.array(lo[:A], np.float32), np.array(hi[:A], np.float32)


def hold_setup(bounds, nan=False):
    """A policy that holds on part of the env-steps: zero pi network, the hold action as output bias, a tiny std except on
    component 0, whose std is the width of its hold interval.  `nan`: one NaN output bias (the action error).
    Returns (setup(policy, client), can_hold)."""
    head, can_hold = orc.hold_action(bounds or {})

    def setup(policy, client):
        lo, hi = hold_intervals(client)
        with torch.no_grad():
            for p_ in policy.pi.parameters():
                p_.zero_()
            policy.pi[4].bias.copy_(torch.as_tensor(head))
            policy.log_std.fill_(-40.0)
            policy.log_std[0] = math.log(max(float(hi[0]) - float(lo[0]), 1e-30))
            if nan:
                policy.pi[4].bias[head.size - 1] = float("nan")
    return setup, bool(np.all(can_hold))


class Case:
    """A handle of a robot with its oracle and an fp32 fused-rollout collector over MlpPolicy(3J, A), the population
    prepared and snapshotted."""

    def __init__(self, bounds, flags=None, n=3001, T=6, seed=31, env_id_base=0, setup=None, f64=False, prepare=True,
                 env=None):
        from gym_roboy_b200.rollout import MlpPolicy, RolloutCollector
        self.bounds, self.flags, self.n, self.T, self.seed = bounds, dict(flags or {}), n, T, seed
        self.env_id_base, self.f64 = env_id_base, f64
        self.env_vars = dict(ROBOY_B200_PENALTY_F64="1" if f64 else "0", **(env or {}))
        with environ(**self.env_vars):
            self.env, self.client, self.ora = make(n, seed, bounds, env_id_base=env_id_base, **self.flags)
            J, A = self.client.dim_obs // 3, self.client.dim_action
            torch.manual_seed(0)
            self.policy = MlpPolicy(3 * J, A).to(DEV)
            with torch.no_grad():
                self.policy.log_std.copy_(torch.linspace(-1.0, 0.7, A))   # a few actions beyond [-1, 1]: clipped
            if setup is not None:
                setup(self.policy, self.client)
            self.col = RolloutCollector(self.env, self.policy, n_steps=T, fused="fp32", noise_seed=NOISE_SEED)
        self.J, self.A = J, A
        self.col.noise = torch.zeros((T, n, A), dtype=torch.float32, device=DEV)
        self.ora.reset()
        if prepare:
            self.prepare()
        self.sd = self.client.state_dict()
        self.obs0 = self.col.obs[0].clone()

    def prepare(self):
        rng = np.random.default_rng(self.seed)
        n = self.n
        steps = rng.integers(1, 401, n)
        cluster = rng.random(n) < 0.2
        steps[cluster] = rng.integers(395, 401, int(cluster.sum()))   # timeouts inside the launch
        set_phases(self.client, self.ora, steps)
        held = np.sort(rng.choice(n, max(n // 50, 1), replace=False))
        feasible = rng.random(held.size) < 0.5
        inject_held(self.client, self.ora, rng, held, feasible)
        J, fast = self.J, held[1::3]
        q, qd = self.ora.held[:J, fast].T.copy(), np.full((fast.size, J), 1e3, np.float32)
        self.client.set_state(q, qd, feasible[1::3].astype(np.uint8), idx=fast)
        self.ora.held[J:, fast] = qd.T
        plant_goals(self.client, self.ora, rng, self.seed, self.T, held, midpoints=True)

    def collect(self):
        self.col.collect()
        torch.cuda.synchronize()

    def twin(self, **env):
        with environ(**dict(self.env_vars, **env)):
            _, c, _ = make(self.n, self.seed, self.bounds, env_id_base=self.env_id_base, **self.flags)
        c.load_state_dict(self.sd)
        return c


def check_policy(case, t0):
    """values, mean + std * z and logp against the torch float32 policy; the noise against its definition."""
    col, policy, T, A = case.col, case.policy, case.T, case.A
    std = policy.log_std.detach().exp()
    lognorm = -0.5 * math.log(2 * math.pi) * A - float(policy.log_std.detach().sum())
    gids = np.arange(case.n, dtype=np.uint64) + np.uint64(case.env_id_base)
    with torch.no_grad():
        for t in range(T + 1):
            mean, value = policy(col.obs[t] if t else case.obs0)
            fin = torch.isfinite(value)
            assert torch.allclose(col.values[t][fin], value[fin], **TOL), t
            if t == T:
                break
            z = col.noise[t]
            want = mean + std * z
            assert torch.allclose(col.actions[t], want, equal_nan=True, **TOL), t
            assert torch.allclose(col.logp[t], lognorm - 0.5 * (z * z).sum(-1), rtol=1e-5, atol=1e-4), t
            assert np.allclose(z.cpu().numpy(), numpy_noise(NOISE_SEED, gids, t0 + 1 + t, A), rtol=0, atol=2e-4), t


def run_case(case, nan=False, expect_holds=True):
    client, ora, col, T, n = case.client, case.ora, case.col, case.T, case.n
    m, _, _ = policy_m(client, "fp32", 0, T)
    tally = Tally(client, ora)
    t0 = client.counter
    case.collect()
    assert not client.msj_kernels
    assert client.counter == t0 + T
    if not nan:
        check_policy(case, t0)

    # ---- the CPU oracle on the clipped actions ----
    acts = np.clip(col.actions.cpu().numpy(), -1.0, 1.0)
    obs, rew, done = col.obs.cpu().numpy(), col.rewards.cpu().numpy(), col.dones.cpu().numpy()
    holds = ora.stats()["holds"]
    for t in range(T):
        o, r, d = ora.step(acts[t])
        check_outputs(obs[t + 1], rew[t], done[t], o, r, d, t)
    holds = ora.stats()["holds"] - holds
    check_state(client, ora)
    assert errors_equal(client.errors(), ora.errors()), (client.errors(), ora.errors())
    tally.check(col.rewards, m)
    if expect_holds and not nan:
        assert 0 < holds < n * T, holds
    assert ora.stats()["episodes"] > 0

    # ---- the generic step kernel on a second handle: bit for bit ----
    k = case.twin()
    assert not k.msj_kernels
    replay_on_step_kernel(k, col, T, bitwise)
    same_env_state(k, client)
    k.close()
    return case


FLAGS = {"default": dict(), "penalty": dict(penalty=True), "nobonus": dict(bonus=False), "manual_reset": dict(auto_reset=False)}


@pytest.mark.parametrize("flags", sorted(FLAGS))
@pytest.mark.parametrize("name", sorted(GENERIC_ROBOTS))
def test_generic_robots_in_the_fused_rollout(name, flags):
    """Every generic robot (per_component_msj_dims has MSJ's dims but per-component bounds: it runs generic) under
    every flag; n = 3001 leaves a ragged tail and unaligned obs slices for even and odd 3J."""
    b = GENERIC_ROBOTS[name]
    setup, can_hold = hold_setup(b)
    run_case(Case(b, FLAGS[flags], setup=setup), expect_holds=can_hold)


def test_float64_penalty_handle_in_the_fused_rollout():
    b = GENERIC_ROBOTS["six_joints_14_tendons"]
    setup, _ = hold_setup(b)
    c32, c64 = (Case(b, dict(penalty=True), setup=setup, f64=f64) for f64 in (False, True))
    assert c32.client.penalty_float32 and not c64.client.penalty_float32
    run_case(c64)
    c32.collect()
    a, b_ = c32.col, c64.col
    assert torch.equal(a.actions, b_.actions) and torch.equal(a.obs, b_.obs) and torch.equal(a.dones, b_.dones)
    r32, r64 = a.rewards.double(), b_.rewards.double()
    assert ((r32 - r64).abs() <= PENALTY_REL * r64.abs()).all()


@pytest.mark.parametrize("J", list(range(1, 16)))
def test_every_joint_count_instantiation(J):
    """generic_policy_rollout_kernel<J> on a random robot (asymmetric per-component bounds, random tendon count), the
    penalty on odd J, global env ids from 777 on even J."""
    rng = np.random.default_rng(2000 + J)
    b = random_robot(rng, J)
    run_case(Case(b, dict(penalty=bool(J % 2)), n=1000 + 37 * J, T=5, seed=J, env_id_base=0 if J % 2 else 777),
             expect_holds=False)


@pytest.mark.parametrize("n", [70_001])
def test_warps_walk_several_chunks(n):
    b = GENERIC_ROBOTS["fifteen_joints_64_tendons"]
    setup, can_hold = hold_setup(b)
    case = Case(b, dict(penalty=True), n=n, T=3, setup=setup)
    m, _, _ = policy_m(case.client, "fp32", 0, case.T)
    assert m >= 2 * case.T   # some warp walks two chunks or more
    run_case(case, expect_holds=can_hold)


def test_step_counter_cap_inside_the_launch():
    b = GENERIC_ROBOTS["six_joints_14_tendons"]
    case = Case(b, dict(auto_reset=False), n=2003, T=4, prepare=False)
    n = case.n
    set_phases(case.client, case.ora, np.where(np.arange(n) % 2 == 0, CAP - 1, CAP))
    rng = np.random.default_rng(3)
    idx = np.flatnonzero(np.arange(n) % 3 == 0)
    inject_held(case.client, case.ora, rng, idx, rng.random(idx.size) < 0.5)
    case.sd = case.client.state_dict()
    case.obs0 = case.col.obs[0].clone()
    run_case(case, expect_holds=False)
    assert case.client.stats()["sum_episode_len"] > 2 ** 32


@pytest.mark.parametrize("name", ["six_joints_14_tendons", "fifteen_joints_64_tendons", "five_joints_11_tendons_per_component"])
def test_nan_weight_trips_the_action_error(name):
    b = GENERIC_ROBOTS[name]
    setup, _ = hold_setup(b, nan=True)
    case = run_case(Case(b, setup=setup, n=2001), nan=True)
    flags, first = case.client.errors()
    assert flags & orc.ERR_ACTION and first == 0
    assert torch.isnan(case.col.actions[:, :, case.A - 1]).all()


# ------------------------------------------------------------------------------------ MSJ through the generic rollout
@pytest.mark.parametrize("penalty", [False, True])
def test_msj_forced_through_the_generic_rollout_equals_the_msj_kernel(penalty):
    """The same seeds, policy and population on K5 and on the generic rollout: everything bit for bit (rewards within
    rewards_agree's tolerance under the penalty, where the two step implementations may differ in the last float32
    bits of the float32-evaluated penalty)."""
    setup, _ = hold_setup(None)
    k5 = Case(None, dict(penalty=penalty), n=6001, T=6, setup=setup)
    gen = Case(None, dict(penalty=penalty), n=6001, T=6, setup=setup, env=dict(ROBOY_B200_FORCE_GENERIC="1"))
    assert k5.client.msj_kernels and not gen.client.msj_kernels
    for c in (k5, gen):
        c.collect()
    a, b = k5.col, gen.col
    for what in ("actions", "logp", "values", "noise", "obs", "dones"):
        assert torch.equal(getattr(a, what).view(torch.int32) if getattr(a, what).dtype == torch.float32 else getattr(a, what),
                           getattr(b, what).view(torch.int32) if getattr(b, what).dtype == torch.float32 else getattr(b, what)), what
    assert rewards_agree(a.rewards, b.rewards, penalty, "float32")
    if not penalty:
        assert bitwise(a.rewards, b.rewards)
    same_env_state(k5.client, gen.client)


# ------------------------------------------------------------------------------------------------------------ invariants
def test_two_half_shards_equal_one_full_shard():
    b = GENERIC_ROBOTS["five_joints_11_tendons_per_component"]
    n, half = 4000, 2000
    full = Case(b, n=n, prepare=False)
    lo = Case(b, n=half, prepare=False)
    hi = Case(b, n=half, env_id_base=half, prepare=False)
    for c in (full, lo, hi):
        c.collect()
    for what in ("actions", "logp", "values", "obs", "rewards", "dones", "noise"):
        f = getattr(full.col, what)
        assert torch.equal(f[:, :half], getattr(lo.col, what)) and torch.equal(f[:, half:], getattr(hi.col, what)), what


def test_cuda_graph_replays_equal_eager_collection():
    b = GENERIC_ROBOTS["six_joints_14_tendons"]
    g, e = Case(b, n=3001, prepare=False), Case(b, n=3001, prepare=False)
    g.col.capture()   # runs one eager warm-up rollout: bring the eager twin to the same point
    e.collect()
    for _ in range(2):
        g.col.collect()
        e.col.collect()
        torch.cuda.synchronize()
        for what in ("actions", "obs", "rewards", "dones", "values", "logp", "adv"):
            assert torch.equal(getattr(g.col, what), getattr(e.col, what)), what


def test_resumed_collector_continues_bit_for_bit():
    b = GENERIC_ROBOTS["fifteen_joints_64_tendons"]
    a = Case(b, n=2001, prepare=False)
    a.collect()
    sd = a.col.state_dict()
    a.collect()
    r = Case(b, n=2001, prepare=False)
    r.col.load_state_dict(sd)
    r.collect()
    for what in ("actions", "obs", "rewards", "dones", "values", "adv", "ret"):
        assert torch.equal(getattr(a.col, what), getattr(r.col, what)), what


def test_tensor_core_modes_refuse_other_robots():
    from gym_roboy_b200 import _native
    from gym_roboy_b200.rollout import MlpPolicy, RolloutCollector
    b = GENERIC_ROBOTS["six_joints_14_tendons"]
    env, client, _ = make(64, 1, b)
    policy = MlpPolicy(18, 14).to(DEV)
    for fused in (True, "tc", "tc_exact"):
        with pytest.raises(ValueError, match='fused="fp32"'):
            RolloutCollector(env, policy, n_steps=2, fused=fused)
    buf = torch.zeros(1 << 16, dtype=torch.float32, device=DEV)
    p = ctypes.c_void_p(buf.data_ptr())
    rc = _native.load().roboy_policy_rollout_tc(client._h, 2, p, 0, p, p, p, p, p, p, None, 0, 0, None)
    assert rc == -1 and b"roboy_policy_rollout" in _native.load().roboy_last_error()


def test_rollout_and_geometry_agree_on_envs_per_thread():
    """Robots other than MSJ run one env per thread: roboy_policy_rollout and roboy_policy_geometry both refuse 2 and
    both take 0 and 1 (the same geometry)."""
    from gym_roboy_b200 import _native
    lib = _native.load()
    _, client, _ = make(5000, 1, GENERIC_ROBOTS["six_joints_14_tendons"])
    buf = torch.zeros(1 << 20, dtype=torch.float32, device=DEV)
    p = ctypes.c_void_p(buf.data_ptr())
    out = [ctypes.c_int() for _ in range(4)]
    assert lib.roboy_policy_geometry(client._h, 2, *(ctypes.byref(o) for o in out)) == -1
    assert lib.roboy_policy_rollout(client._h, 1, p, 0, p, p, p, p, p, p, None, 2, None) == -1
    geo = []
    for ept in (0, 1):
        _native.check(lib.roboy_policy_geometry(client._h, ept, *(ctypes.byref(o) for o in out)))
        geo.append([o.value for o in out])
    assert geo[0] == geo[1] and geo[0][3] == 1 and geo[0][1] <= 256
