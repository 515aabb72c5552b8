"""Deterministic policy evaluation (`roboy_policy_evaluate`, roboy_policy_eval.cu; `gym_roboy_b200.evaluation`).

The main comparison runs the evaluator on a second handle with the same prepared population as a reference: the float32
fused rollout (`RolloutCollector(fused="fp32")`) for the same T steps with log_std = -200, whose float32 std is exactly 0,
so that its env outputs are those of the policy mean.  From the reference's rewards, dones and initial step counters a
numpy restatement of the counting rule derives every record (float64 returns summed in step order), `completed` and
the final observation; the evaluator must give the same bits.  Goals, step words, error word, first offender and the
statistics counts must equal the reference's.  The `reached` flags, which the reference does not store, are checked
against the handle's own statistics in runs where every finished episode is recorded, and on goals planted to be
reached on the timeout step.
"""
import ctypes
import math

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from test_gpu_episode_stats import make
from test_gpu_generic_robots import PENALTY_REL
from test_gpu_policy_rollout_envs import same_env_state
from test_gpu_policy_rollout_generic import Case, hold_setup
from test_oracle_vs_reference import GENERIC_ROBOTS, random_robot

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
MASK = orc.STEP_MASK
L = 400   # max_episode_len of every handle here (roboy_env.py:28)


def std0(inner=None):
    """A Case setup: `inner`'s policy, then log_std = -200, whose exp is 0 in float32 (the rollout's action = the mean)."""
    def setup(policy, client):
        if inner is not None:
            inner(policy, client)
        with torch.no_grad():
            policy.log_std.fill_(-200.0)
            assert float(policy.log_std.exp().max()) == 0.0
    return setup


def native():
    from gym_roboy_b200 import _native
    return _native, _native.load()


def image_of(policy, client):
    from gym_roboy_b200.rollout import pack_policy_image
    _native, _ = native()
    img = torch.zeros(_native.policy_layout(client.dim_obs, client.dim_action)[_native.POLICY_LAYOUT_FLOATS],
                      dtype=torch.float32, device=DEV)
    return pack_policy_image(policy, out=img)


def evaluate(client, image, T, K, obs, fill=None):
    """roboy_policy_evaluate on the whole handle; returns (returns, lengths, reached, completed) as device tensors."""
    _native, lib = native()
    n = client.num_envs
    returns = torch.full((K, n), 7.0 if fill is None else fill, dtype=torch.float64, device=DEV)   # no return is +7
    lengths = torch.full((K, n), 0x5A5A5A5A, dtype=torch.int32, device=DEV)
    reached = torch.full((K, n), 0x77, dtype=torch.uint8, device=DEV)
    completed = torch.full((n,), -1, dtype=torch.int32, device=DEV)
    p = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
    _native.check(lib.roboy_policy_evaluate(client._h, T, p(image), p(obs), K, p(returns), p(lengths), p(reached),
                                            p(completed), None))
    torch.cuda.synchronize()
    return returns, lengths, reached, completed


def implied_records(sf0, rewards, dones, K):
    """The counting rule restated in numpy: from the initial step words and the per-step rewards / dones, the records
    [K][n] (returns float64 summed in step order, lengths, a filled mask) and completed [n]."""
    T, n = rewards.shape
    s = (sf0.astype(np.int64) & MASK)
    counting = s == 1
    ret = np.zeros(n)
    n_rec = np.zeros(n, np.int64)
    n_done = np.zeros(n, np.int64)
    R = np.full((K, n), np.nan)
    Ln = np.zeros((K, n), np.int64)
    absum, Ab = np.zeros(n), np.zeros((K, n))   # sum |r| of each record (the tolerance of MSJ's penalty rewards)
    for t in range(T):
        s = s + (s < MASK)
        d = dones[t].astype(bool)
        ret = np.where(counting, ret + rewards[t].astype(np.float64), ret)
        absum = np.where(counting, absum + np.abs(rewards[t].astype(np.float64)), absum)
        rec = counting & d
        w = np.flatnonzero(rec & (n_rec < K))
        R[n_rec[w], w] = ret[w]
        Ln[n_rec[w], w] = s[w] - 1
        Ab[n_rec[w], w] = absum[w]
        n_rec[w] += 1
        n_done += rec
        counting = counting | d
        ret[d] = absum[d] = 0.0
        s[d] = 1
    return R, Ln, n_rec, n_done, Ab


def check_records(out, R, Ln, n_rec, n_done, Ab, rtol=0.0):
    returns, lengths, reached, completed = (t.cpu().numpy() for t in out)
    K = R.shape[0]
    filled = np.arange(K)[:, None] < n_rec[None, :]
    assert np.array_equal(np.isnan(returns), ~filled)
    if rtol:
        assert np.all(np.abs(returns[filled] - R[filled]) <= rtol * Ab[filled])
    else:
        assert np.array_equal(returns.view(np.int64), R.view(np.int64))   # bit for bit, NaNs included
    assert np.array_equal(lengths.astype(np.int64), Ln)
    assert np.all(reached[~filled] == 0) and np.all(reached <= 1)
    assert np.array_equal(completed.astype(np.int64), n_done)
    # a done before the timeout comes from _did_reach_goal
    assert np.all(reached[filled & (Ln < L)] == 1)


def count_from_reset(client, frac, seed):
    """Step counter 1 (the reset value) on a fraction of the envs: their first episode counts from call 1."""
    rng = np.random.default_rng(seed)
    idx = np.flatnonzero(rng.random(client.num_envs) < frac)
    client.set_step_num(np.ones(idx.size, np.int32), idx=idx)


def compare(bounds, flags=None, n=3001, T=8, K=3, seed=31, env_id_base=0, setup=None, msj=False):
    """The evaluator against the std-0 fused rollout on the same prepared population (see the module docstring)."""
    c = Case(bounds, flags, n=n, T=T, seed=seed, env_id_base=env_id_base, setup=std0(setup))
    count_from_reset(c.client, 0.3, seed)
    c.sd = c.client.state_dict()
    sf0 = c.client.step_flags.cpu().numpy().astype(np.uint32)
    k = c.twin()
    image = image_of(c.policy, k)
    obs = c.obs0.clone()
    t0, s0 = k.counter, k.stats()
    out = evaluate(k, image, T, K, obs)
    assert k.counter == t0 + T
    c.collect()
    assert k.msj_kernels == c.client.msj_kernels == msj
    rew, done = c.col.rewards.cpu().numpy(), c.col.dones.cpu().numpy()
    rec = implied_records(sf0, rew, done, K)
    penalty = bool((flags or {}).get("penalty"))
    # MSJ under the penalty: the reference ran K5, whose rewards agree with the generic step's to PENALTY_REL
    check_records(out, *rec, rtol=2 * PENALTY_REL if (msj and penalty) else 0.0)
    assert torch.equal(obs.view(torch.int32), c.col.obs[T].view(torch.int32))
    same_env_state(k, c.client)
    s1, r1 = k.stats(), c.client.stats()
    d_eval, d_ref = s1["sum_reward"] - s0["sum_reward"], r1["sum_reward"] - s0["sum_reward"]
    assert abs(d_eval - d_ref) <= 1e-6 * np.abs(rew).astype(np.float64).sum() + 1e-9
    k.close()
    return c, out, rec


FLAGS = {"default": dict(), "penalty": dict(penalty=True), "nobonus": dict(bonus=False)}
ROBOTS = dict(msj=None, **GENERIC_ROBOTS)


@pytest.mark.parametrize("flags", sorted(FLAGS))
@pytest.mark.parametrize("name", sorted(ROBOTS))
def test_every_robot_against_the_std0_rollout(name, flags):
    """Every generic robot and MSJ under default, penalty and no-bonus; the policy holds wherever it can (the mean is the
    hold action), so that envs counted from call 1 reach goals planted around their state."""
    b = ROBOTS[name]
    setup, _ = hold_setup(b)
    compare(b, FLAGS[flags], setup=setup, msj=name == "msj")


@pytest.mark.parametrize("flags", ["default", "penalty"])
@pytest.mark.parametrize("name", ["msj", "six_joints_14_tendons"])
def test_a_policy_that_does_not_hold(name, flags):
    """The random MlpPolicy's mean: actions spread over [-1, 1], some clipped."""
    compare(ROBOTS[name], FLAGS[flags], T=10, msj=name == "msj")


@pytest.mark.parametrize("J", list(range(1, 16)))
def test_every_joint_count_instantiation(J):
    rng = np.random.default_rng(3000 + J)
    b = random_robot(rng, J)
    compare(b, dict(penalty=bool(J % 2)), n=1000 + 37 * J, T=6, seed=J, env_id_base=0 if J % 2 else 777,
            setup=hold_setup(b)[0] if J % 3 == 0 else None)


def test_ragged_n_non_zero_env_id_base_and_warps_that_walk_several_chunks():
    from test_gpu_episode_stats import policy_m
    b = GENERIC_ROBOTS["fifteen_joints_64_tendons"]
    c, _, _ = compare(b, dict(penalty=True), n=70_001, T=3, K=2, env_id_base=123_457, setup=hold_setup(b)[0])
    m, _, _ = policy_m(c.client, "fp32", 0, c.T)
    assert m >= 2 * c.T   # some warp walks two chunks or more (the evaluator uses the rollout's geometry)


def test_two_half_shards_equal_one_full_shard():
    b = GENERIC_ROBOTS["five_joints_11_tendons_per_component"]
    n, half, T, K = 4000, 2000, 450, 2
    outs = []
    for nn, base in ((n, 0), (half, 0), (half, half)):
        env, client, _ = make(nn, 11, b, env_id_base=base)
        from gym_roboy_b200.evaluation import evaluate_policy
        from gym_roboy_b200.rollout import MlpPolicy
        torch.manual_seed(0)
        policy = MlpPolicy(client.dim_obs, client.dim_action).to(DEV)
        res = evaluate_policy(env, policy, n_eval_episodes=K, n_steps=T)
        outs.append((res, client.obs.clone(), client.goal.clone()))
    full, lo, hi = outs
    bits = lambda t: t.view(torch.int64) if t.dtype == torch.float64 else t   # noqa: E731  (NaN-safe)
    for what in ("returns", "lengths", "reached"):
        f = bits(getattr(full[0], what))
        assert torch.equal(f[:, :half], bits(getattr(lo[0], what))) and torch.equal(f[:, half:], bits(getattr(hi[0], what))), what
    assert torch.equal(full[0].completed, torch.cat([lo[0].completed, hi[0].completed]))
    assert torch.equal(full[1], torch.cat([lo[1], hi[1]]))
    assert torch.equal(full[2], torch.cat([lo[2], hi[2]], dim=1))
    assert int(full[0].completed.sum()) > 0


# ------------------------------------------------------------------------------------------ reached, independently
WIDE_VELS = dict(dim_joint=3, dim_action=5, angle_low=-1.0, angle_high=1.0, vel_low=-10.0, vel_high=10.0, act_low=-0.3,
                 act_high=0.3)   # the Stub draws velocities from the angle space: every sampled state is vels-close


def test_reached_flags_against_the_statistics_when_every_episode_is_recorded():
    """After a reset every episode counts; K >= T records them all: sum(reached) = delta SUCCESSES, sum(lengths) = delta
    SUM_EPLEN, records = delta EPISODES.  Goals planted at the states of steps 1..40 make early reaches."""
    from gym_roboy_b200.evaluation import evaluate_policy
    from gym_roboy_b200.rollout import MlpPolicy
    n, T = 20_000, 450
    env, client, ora = make(n, 7, WIDE_VELS)
    torch.manual_seed(1)
    policy = MlpPolicy(client.dim_obs, client.dim_action).to(DEV)
    env.reset()
    rng = np.random.default_rng(7)
    gids = np.arange(n, dtype=np.uint64)
    k = rng.integers(1, 41, n)
    q = np.zeros((n, 3), np.float32)
    for kk in range(1, 41):
        sel = np.flatnonzero(k == kk)
        q[sel] = orc.draw_state(7, gids[sel], client.counter + kk, ora.bounds["angle_low"], ora.bounds["angle_high"], J=3)[0]
    client.set_goal(q)
    s0 = client.stats()
    res = evaluate_policy(env, policy, n_eval_episodes=T, n_steps=T, reset=False)
    s1 = client.stats()
    rec = ~torch.isnan(res.returns)
    assert int(rec.sum()) == s1["episodes"] - s0["episodes"] == int(res.completed.sum())
    assert int(res.reached.sum()) == s1["successes"] - s0["successes"]
    assert int(res.lengths.long().sum()) == s1["sum_episode_len"] - s0["sum_episode_len"]
    early = res.reached[0].cpu().numpy() & (res.lengths[0].cpu().numpy() == k)
    assert early.mean() > 0.5, early.mean()   # most planted goals are reached on their step
    assert int(res.reached.sum()) < int(rec.sum())   # and timeouts without a reach exist


def test_goal_reached_on_the_timeout_step():
    """Goals planted at the state of step 400 after a reset: the done is a timeout and a reach at once, reached = 1."""
    from gym_roboy_b200.evaluation import evaluate_policy
    from gym_roboy_b200.rollout import MlpPolicy
    n = 4096
    env, client, ora = make(n, 9, WIDE_VELS)
    torch.manual_seed(2)
    policy = MlpPolicy(client.dim_obs, client.dim_action).to(DEV)
    env.reset()
    gids = np.arange(n, dtype=np.uint64)
    planted = np.arange(n) % 2 == 0
    q = orc.draw_state(9, gids, client.counter + L, ora.bounds["angle_low"], ora.bounds["angle_high"], J=3)[0]
    g = client.goal.t().cpu().numpy().copy()
    g[planted] = q[planted]
    client.set_goal(g.astype(np.float32))
    s0 = client.stats()
    res = evaluate_policy(env, policy, n_eval_episodes=1, n_steps=L, reset=False)
    s1 = client.stats()
    lengths, reached = res.lengths[0].cpu().numpy(), res.reached[0].cpu().numpy()
    on_time = planted & (lengths == L)
    assert on_time.sum() > 0.9 * planted.sum()
    assert reached[on_time].all()
    assert s1["successes"] - s0["successes"] == int(res.reached.sum())
    assert s1["timeouts"] - s0["timeouts"] == int(((lengths == L) & (reached == 0)).sum())


# --------------------------------------------------------------------------------------------- the public function
def hold_env(n, seed, name="six_joints_14_tendons"):
    from gym_roboy_b200.rollout import MlpPolicy
    b = GENERIC_ROBOTS[name]
    env, client, _ = make(n, seed, b)
    setup, can_hold = hold_setup(b)
    assert can_hold
    policy = MlpPolicy(client.dim_obs, client.dim_action).to(DEV)
    setup(policy, client)
    return env, client, policy


def test_holding_policy_after_a_reset_gives_exactly_k_timeouts():
    """The env holds at the zero state of reset(): every episode times out, so the default n_steps = K * 400 leaves
    exactly K episodes of length 400 per env, none reached."""
    from gym_roboy_b200.evaluation import evaluate_policy
    env, client, policy = hold_env(4096, 3)
    K = 2
    s0 = client.stats()
    res = evaluate_policy(env, policy, n_eval_episodes=K)
    s1 = client.stats()
    assert res.n_steps == K * L and res.returns.shape == (K, 4096)
    assert (res.completed == K).all() and (res.lengths == L).all() and not res.reached.any()
    assert res.n_episodes == K * 4096 and res.success_rate == 0.0 and res.mean_length == L
    assert s1["holds"] - s0["holds"] == K * L * 4096
    assert math.isclose(res.mean_return, float(res.returns.mean()), rel_tol=1e-12)
    assert math.isclose(res.std_return, float(res.returns.std(unbiased=False)), rel_tol=1e-9, abs_tol=1e-9)


def test_mid_episode_envs_are_not_counted_until_their_next_episode():
    """Without a reset, an env in the middle of an episode finishes it uncounted; the default n_steps (K + 1) * 400
    still gives K counted episodes.  Envs at step 1 count from call 1 (and finish one more)."""
    from gym_roboy_b200.evaluation import evaluate_policy
    n = 4096
    env, client, policy = hold_env(n, 4)
    steps = (np.arange(n) % L + 1).astype(np.int32)   # 1..400
    client.set_step_num(steps)
    res = evaluate_policy(env, policy, n_eval_episodes=1, reset=False)
    assert res.n_steps == 2 * L
    completed = res.completed.cpu().numpy()
    assert np.array_equal(completed, np.where(steps == 1, 2, 1))
    assert (res.lengths[0] == L).all() and not res.reached.any()


def test_k1_records_only_the_first_of_several_episodes():
    from gym_roboy_b200.evaluation import evaluate_policy
    env, client, policy = hold_env(2048, 5)
    res = evaluate_policy(env, policy, n_eval_episodes=1, n_steps=3 * L + 7)
    assert (res.completed == 3).all() and res.returns.shape == (1, 2048)
    assert (res.lengths[0] == L).all() and not torch.isnan(res.returns).any()


def test_env_step_continues_from_the_evaluation():
    """The observation buffer holds the observation after the last step, so env.step continues the same trajectory as
    an uninterrupted evaluation."""
    from gym_roboy_b200.evaluation import evaluate_policy
    from gym_roboy_b200.rollout import MlpPolicy
    b = GENERIC_ROBOTS["six_joints_14_tendons"]
    outs = []
    for split in (False, True):
        env, client, _ = make(3001, 6, b)
        torch.manual_seed(0)
        policy = MlpPolicy(client.dim_obs, client.dim_action).to(DEV)
        if split:
            evaluate_policy(env, policy, n_eval_episodes=0, n_steps=5)
            with torch.no_grad():
                a = torch.clamp(policy.pi(client.obs), -1.0, 1.0).contiguous()
            env.step(a)
            obs_mid = client.obs.clone()
            res = evaluate_policy(env, policy, n_eval_episodes=0, n_steps=4, reset=False)
            outs.append((client.obs.clone(), client.goal.clone(), client.step_flags.clone(), client.counter, obs_mid))
        else:
            res = evaluate_policy(env, policy, n_eval_episodes=0, n_steps=10)
            outs.append((client.obs.clone(), client.goal.clone(), client.step_flags.clone(), client.counter, None))
    assert outs[0][3] == outs[1][3]
    for i in range(3):
        assert torch.equal(outs[0][i], outs[1][i]), i


def test_nan_weight_trips_the_action_error_with_the_reference_offender():
    b = GENERIC_ROBOTS["six_joints_14_tendons"]
    setup, _ = hold_setup(b, nan=True)
    c, _, _ = compare(b, n=2001, setup=setup)
    flags, first = c.client.errors()
    assert flags & orc.ERR_ACTION and first == 0


def test_msj_evaluation_runs_the_generic_step():
    """An MSJ handle evaluates on the generic env step; with the penalty its rewards agree with K1's to PENALTY_REL."""
    c, out, _ = compare(None, dict(penalty=True), n=6001, T=8, setup=hold_setup(None)[0], msj=True)
    assert c.client.msj_kernels


def test_mismatched_policy_fails_in_pack_policy_image():
    from gym_roboy_b200.evaluation import evaluate_policy
    from gym_roboy_b200.rollout import MlpPolicy
    env, client, _ = make(64, 1, GENERIC_ROBOTS["six_joints_14_tendons"])
    with pytest.raises(AssertionError):
        evaluate_policy(env, MlpPolicy().to(DEV), n_eval_episodes=1)


# ------------------------------------------------------------------------------------------------------- refusals
def test_refusals_and_t0():
    _native, lib = native()
    from gym_roboy_b200.rollout import MlpPolicy
    b = GENERIC_ROBOTS["six_joints_14_tendons"]
    _, client, _ = make(256, 1, b)
    img = image_of(MlpPolicy(client.dim_obs, client.dim_action).to(DEV), client)
    buf = torch.zeros(1 << 16, dtype=torch.float64, device=DEV)
    obs = client.obs.clone()
    P = lambda t, off=0: ctypes.c_void_p(t.data_ptr() + off)  # noqa: E731
    args = lambda image, o: (client._h, 3, image, o, 2, P(buf), P(buf), P(buf), P(buf), None)  # noqa: E731
    good = args(P(img), P(obs))
    for i in (0, 2, 3, 5, 6, 7, 8):
        bad = list(good)
        bad[i] = None
        assert lib.roboy_policy_evaluate(*bad) == -1 and b"NULL" in lib.roboy_last_error()
    assert lib.roboy_policy_evaluate(*args(P(img, 4), P(obs))) == -1 and b"16-byte" in lib.roboy_last_error()
    assert lib.roboy_policy_evaluate(*args(P(img), P(obs, 2))) == -1 and b"4-byte" in lib.roboy_last_error()
    # T = 0: no launch, nothing moves
    t0, n0 = client.counter, client.launch_count()
    before = buf.clone()
    assert lib.roboy_policy_evaluate(client._h, 0, P(img), P(obs), 2, P(buf), P(buf), P(buf), P(buf), None) == 0
    torch.cuda.synchronize()
    assert client.counter == t0 and client.launch_count() == n0 and torch.equal(buf, before)
    assert lib.roboy_policy_evaluate(*good) == 0 and client.launch_count() == n0 + 1 and client.counter == t0 + 3
    # auto_reset off: no new episode would ever start
    _, manual, _ = make(256, 1, b, auto_reset=False)
    assert lib.roboy_policy_evaluate(manual._h, 3, P(img), P(obs), 2, P(buf), P(buf), P(buf), P(buf), None) == -1
    assert b"auto_reset" in lib.roboy_last_error()


# ------------------------------------------------------------------------------------------------- 64-bit offsets
def test_record_arrays_past_4_gib():
    """K * n > 2^32 slots (the reached array alone is past 4 GiB): a handle with max_episode_len = 1 finishes an
    episode on every step, so after T = K steps every slot up to the last is written."""
    _native, lib = native()
    from gym_roboy_b200.rollout import MlpPolicy
    free, _ = torch.cuda.mem_get_info()
    n, K = 1 << 22, 1025
    assert K * n > 1 << 32
    if free < 70e9:
        pytest.skip("needs ~56 GB of free device memory")
    cfg = _native.RoboyCfg()
    _native.check(lib.roboy_cfg_msj(ctypes.byref(cfg)))
    cfg.n_envs, cfg.seed, cfg.max_episode_len = n, 1, 1
    h = ctypes.c_void_p()
    _native.check(lib.roboy_create(ctypes.byref(cfg), 0, ctypes.byref(h)))
    try:
        obs = torch.zeros((n, 9), dtype=torch.float32, device=DEV)
        _native.check(lib.roboy_reset(h, None, ctypes.c_void_p(obs.data_ptr()), None))

        class _C:   # just enough of a client for image_of / evaluate
            _h, num_envs, dim_obs, dim_action = h, n, 9, 8
        torch.manual_seed(0)
        img = image_of(MlpPolicy().to(DEV), _C)
        returns, lengths, reached, completed = evaluate(_C, img, K, K, obs)
        assert (completed == K).all()
        assert (lengths == 1).all()
        assert not torch.isnan(returns).any() and not (returns == 7.0).any()   # every slot written
        assert (reached <= 1).all()
        assert lengths[K - 1, n - 1].item() == 1 and math.isfinite(returns[K - 1, n - 1].item())
        del returns, lengths, reached
        st = (ctypes.c_double * 8)()
        _native.check(lib.roboy_stats(h, st, None))
        assert st[1] == K * n and st[5] == K * n
    finally:
        lib.roboy_destroy(h)
        torch.cuda.empty_cache()
