"""PPO2 minibatch gradient (`roboy_ppo_grad`, roboy_ppo.cu; `gym_roboy_b200.ppo`).

The reference is stable-baselines 2's PPO2 loss restated in torch autograd (`reference` below), run in float64 and in
float32 on the same minibatch.  The kernel's error against float64 must stay within 8 times float32 autograd's error plus
2e-6 of the largest float64 gradient, for every parameter tensor.  Minibatches come from real fused-rollout buffers;
the policy is then perturbed so that ratios and value changes fall on both sides of the clip ranges, and samples whose
ratio or value change lies within 1e-4 of a clip boundary are left out, so float32 and float64 take the same branch of
every max / clip.
"""
import copy
import ctypes
import math

import numpy as np
import pytest
import torch

from test_gpu_episode_stats import robot_from_bounds
from test_oracle_vs_reference import GENERIC_ROBOTS, random_robot

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
ROBOTS = {"msj": None, **{k: GENERIC_ROBOTS[k] for k in ("six_joints_14_tendons", "five_joints_11_tendons_per_component",
                                                         "fifteen_joints_64_tendons")}}
PARAMS = ("vf.0.weight", "vf.0.bias", "vf.2.weight", "vf.2.bias", "vf.4.weight", "vf.4.bias",
          "pi.0.weight", "pi.0.bias", "pi.2.weight", "pi.2.bias", "pi.4.weight", "pi.4.bias", "log_std")


def collected(bounds, n=4096, T=8, seed=3, fused="fp32", fit_value=False):
    """A collector of this robot after one fused rollout (weights as collected).  fit_value: first a rollout to measure
    the mean reward r, then the value net's output bias set to r / (1 - gamma), the value of a steady stream of r, and
    the rollout the minibatches come from: its returns then lie on both sides of the values (with the untrained value
    net near 0 and negative rewards, every return lies below its value)."""
    from gym_roboy_b200.envs import RoboyEnv
    from gym_roboy_b200.envs.simulations import CudaSimulationClient
    from gym_roboy_b200.rollout import MlpPolicy, RolloutCollector
    client = CudaSimulationClient(robot=robot_from_bounds(bounds), num_envs=n, seed=seed, device=DEV)
    env = RoboyEnv(client, strict=False)
    torch.manual_seed(seed)
    policy = MlpPolicy(client.dim_obs, client.dim_action).to(DEV)
    with torch.no_grad():
        policy.log_std.copy_(torch.linspace(-1.0, 0.3, client.dim_action))
    col = RolloutCollector(env, policy, n_steps=T, fused=fused, noise_seed=seed)
    if fit_value:
        col.collect()
        with torch.no_grad():
            policy.vf[4].bias.fill_(float(col.rewards.mean()) / (1.0 - col.gamma))
    obs0 = col.obs[0].clone()
    col.collect()
    col.obs[0].copy_(obs0)     # collect() leaves the next start there; the minibatches need this rollout's
    torch.cuda.synchronize()
    return col


def buffers(col):
    T, N = col.T, col.N
    return (col.obs[:T].reshape(T * N, -1).contiguous(), col.actions.reshape(T * N, -1).contiguous(),
            col.logp.reshape(-1).contiguous(), col.values[:T].reshape(-1).contiguous(), col.ret.reshape(-1).contiguous())


def perturb(policy, scale=0.06, seed=1):
    g = torch.Generator(device="cpu").manual_seed(seed)
    with torch.no_grad():
        for q in policy.parameters():
            q.add_((torch.randn(q.shape, generator=g) * scale).to(q.device))


def reference(policy, bufs, idx, clip=0.2, clip_vf=None, ent_coef=0.01, vf_coef=0.5, dtype=torch.float64):
    """stable-baselines 2's PPO2 loss in torch autograd at `dtype`: returns ({name: grad}, {stat: value})."""
    obs, actions, logp, values, ret = bufs
    p = copy.deepcopy(policy).to(dtype)
    idx = idx[(idx >= 0) & (idx < obs.shape[0])]
    o, a, lp_old, v_old, R = (t[idx].to(dtype) for t in (obs, actions, logp, values, ret))
    adv = (ret[idx] - values[idx]).to(dtype)                 # float32 subtraction, as SB2's numpy
    adv_mean, adv_std = adv.mean(), adv.std(unbiased=False)
    adv = (adv - adv_mean) / (adv_std + 1e-8)
    mean, v = p.pi(o), p.vf(o).squeeze(-1)
    A = mean.shape[-1]
    z = (a - mean) / p.log_std.exp()
    lp = -0.5 * (z * z).sum(-1) - 0.5 * A * math.log(2 * math.pi) - p.log_std.sum()
    ratio = torch.exp(lp - lp_old)
    pg1, pg2 = -adv * ratio, -adv * torch.clamp(ratio, 1 - clip, 1 + clip)
    pg = torch.where(pg1 >= pg2, pg1, pg2).mean()
    e = clip if clip_vf is None else clip_vf
    l1 = (v - R) ** 2
    if e < 0:
        vf = 0.5 * l1.mean()
    else:
        l2 = (v_old + torch.clamp(v - v_old, -e, e) - R) ** 2
        vf = 0.5 * torch.where(l1 >= l2, l1, l2).mean()
    ent = (p.log_std + 0.5 * math.log(2 * math.pi * math.e)).sum()
    loss = pg - ent_coef * ent + vf_coef * vf
    loss.backward()
    grads = {k: q.grad.detach().double() for k, q in p.named_parameters()}
    stats = dict(loss=loss.item(), pg_loss=pg.item(), vf_loss=vf.item(), entropy=ent.item(),
                 approxkl=(0.5 * ((lp - lp_old) ** 2).mean()).item(),
                 clipfrac=((ratio - 1).abs() > clip).double().mean().item(), adv_mean=adv_mean.item(),
                 adv_std=adv_std.item())
    return grads, stats, ratio.detach(), (v - v_old).detach()


def away_from_boundaries(policy, bufs, idx, clip=0.2, clip_vf=None):
    """idx without the samples whose float64 ratio or value change lies within 1e-4 of a clip boundary."""
    _, _, ratio, dv = reference(policy, bufs, idx, clip, clip_vf)
    e = clip if clip_vf is None else clip_vf
    keep = ((ratio - (1 - clip)).abs() > 1e-4) & ((ratio - (1 + clip)).abs() > 1e-4)
    if e >= 0:
        keep &= ((dv - e).abs() > 1e-4) & ((dv + e).abs() > 1e-4)
    return idx[keep].contiguous()


def kernel(policy, bufs, idx, clip=0.2, clip_vf=None, ent_coef=0.01, vf_coef=0.5):
    from gym_roboy_b200.ppo import ppo_grad, unpack_policy_grad
    from gym_roboy_b200.rollout import pack_policy_image
    from gym_roboy_b200 import _native
    image = pack_policy_image(policy)
    grad, stats = ppo_grad(image, *bufs, idx, clip, clip_vf, ent_coef, vf_coef)
    q = copy.deepcopy(policy)
    unpack_policy_grad(q, grad)
    torch.cuda.synchronize()
    return ({k: t.grad.detach().double() for k, t in q.named_parameters()},
            dict(zip(_native.PPO_STAT_NAMES, stats.tolist())), grad)


def check_against_float64(policy, bufs, idx, **kw):
    g64, s64, _, _ = reference(policy, bufs, idx, dtype=torch.float64, **kw)
    g32, _, _, _ = reference(policy, bufs, idx, dtype=torch.float32, **kw)
    gk, sk, grad = kernel(policy, bufs, idx, **kw)
    for name in PARAMS:
        err_k = float((gk[name] - g64[name]).abs().max())
        err_32 = float((g32[name] - g64[name]).abs().max())
        scale = float(g64[name].abs().max())
        assert err_k <= 8 * err_32 + 2e-6 * scale, (name, err_k, err_32, scale)
    for k, r in s64.items():
        if k == "clipfrac":
            assert sk[k] == r, (k, sk[k], r)
        else:
            assert abs(sk[k] - r) <= 1e-5 * abs(r) + 1e-12, (k, sk[k], r)
    assert sk["bad_indices"] == 0
    return gk, sk, grad


def shuffled(col, m=None, seed=0):
    n = col.T * col.N
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randperm(n, generator=g, device=DEV)[: (m or n)].contiguous()


@pytest.fixture(scope="module")
def msj():
    col = collected(None)
    perturb(col.policy)
    return col


@pytest.fixture(scope="module")
def msj_fitted():
    col = collected(None, fit_value=True)
    perturb(col.policy)
    return col


@pytest.mark.parametrize("robot", list(ROBOTS))
def test_gradients_match_float64(robot):
    col = collected(ROBOTS[robot])
    perturb(col.policy)
    bufs = buffers(col)
    idx = away_from_boundaries(col.policy, bufs, shuffled(col))
    _, s, _ = check_against_float64(col.policy, bufs, idx)
    _, _, ratio, _ = reference(col.policy, bufs, idx)
    adv = (bufs[4] - bufs[3])[idx]
    adv = adv - adv.mean()
    # every branch of the surrogate is exercised: ratio clipped above and below, with both advantage signs
    for side in (ratio > 1.2, ratio < 0.8):
        assert bool((side & (adv > 0)).any()) and bool((side & (adv < 0)).any())


@pytest.mark.parametrize("J", list(range(1, 16)))
def test_every_joint_count_instantiation(J):
    col = collected(random_robot(np.random.default_rng(100 + J), J), n=1024, T=4, seed=J)
    perturb(col.policy)
    bufs = buffers(col)
    check_against_float64(col.policy, bufs, away_from_boundaries(col.policy, bufs, shuffled(col)))


@pytest.mark.parametrize("kw", [dict(clip_vf=-1.0), dict(clip_vf=0.05), dict(ent_coef=0.0), dict(clip=0.1, vf_coef=1.0)],
                         ids=["value_clip_off", "own_value_clip", "no_entropy", "other_coefs"])
def test_loss_variants(msj_fitted, kw):
    col = msj_fitted
    bufs = buffers(col)
    idx = away_from_boundaries(col.policy, bufs, shuffled(col), kw.get("clip", 0.2), kw.get("clip_vf"))
    check_against_float64(col.policy, bufs, idx, **kw)
    # the value loss sees returns above and below the new values, so either argument of its max can win
    with torch.no_grad():
        v = col.policy.vf(bufs[0][idx]).squeeze(-1)
    above = bufs[4][idx] > v
    assert 0.1 < float(above.float().mean()) < 0.9


@pytest.mark.parametrize("m", [1, 257, 4_194_304])
def test_minibatch_sizes_with_repeats(msj, m):
    bufs = buffers(msj)
    pool = away_from_boundaries(msj.policy, bufs, shuffled(msj))
    g = torch.Generator(device=DEV).manual_seed(m)
    idx = pool[torch.randint(0, pool.numel(), (m,), generator=g, device=DEV)].contiguous()   # repeats when m > pool
    if m == 257:
        idx[100:120] = idx[5]
    check_against_float64(msj.policy, bufs, idx)


def test_padding_and_lognorm_slot_are_zero():
    from gym_roboy_b200 import _native
    col = collected(GENERIC_ROBOTS["six_joints_14_tendons"], n=1024, T=4)
    perturb(col.policy)
    bufs = buffers(col)
    _, _, grad = kernel(col.policy, bufs, shuffled(col))
    off = _native.policy_layout(col.client.dim_obs, col.client.dim_action)
    A, H = col.client.dim_action, _native.POLICY_HIDDEN
    vf, pi = off[_native.POLICY_LAYOUT_VF], off[_native.POLICY_LAYOUT_PI]
    w3, b3v, b3p = off[_native.POLICY_LAYOUT_W3], off[_native.POLICY_LAYOUT_VF_B3], off[_native.POLICY_LAYOUT_PI_B3]
    g = grad.cpu()
    assert torch.all(g[vf + w3: vf + b3v].view(H, 8)[:, 1:] == 0) and torch.all(g[vf + b3v + 1: vf + b3v + 8] == 0)
    assert torch.all(g[pi + w3: pi + b3p].view(H, 16)[:, A:] == 0) and torch.all(g[pi + b3p + A: pi + b3p + 16] == 0)
    s = off[_native.POLICY_LAYOUT_STD]
    assert torch.all(g[s + A: off[_native.POLICY_LAYOUT_FLOATS]] == 0)
    assert torch.isfinite(g).all() and (g[pi + w3: pi + b3p].view(H, 16)[:, :A] != 0).any()


def test_deterministic_across_calls_and_graph_replay(msj):
    from gym_roboy_b200.ppo import ppo_grad
    from gym_roboy_b200.rollout import pack_policy_image
    bufs = buffers(msj)
    idx = shuffled(msj, 20_000)
    image = pack_policy_image(msj.policy)
    a = [t.clone() for t in ppo_grad(image, *bufs, idx)]
    b = [t.clone() for t in ppo_grad(image, *bufs, idx)]
    grad, stats = torch.empty_like(image), torch.empty(9, dtype=torch.float64, device=DEV)
    ws = torch.empty(10 << 20, dtype=torch.uint8, device=DEV)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ppo_grad(image, *bufs, idx, grad=grad, stats=stats, workspace=ws)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        ppo_grad(image, *bufs, idx, grad=grad, stats=stats, workspace=ws)
    grad.zero_(); stats.zero_()
    graph.replay()
    torch.cuda.synchronize()
    for x in (b, [grad, stats]):
        assert torch.equal(a[0].view(torch.int32), x[0].view(torch.int32))
        assert torch.equal(a[1].view(torch.int64), x[1].view(torch.int64))


def test_buffers_past_4_gib_equal_a_small_gather(msj):
    from gym_roboy_b200.ppo import ppo_grad
    from gym_roboy_b200.rollout import pack_policy_image
    small = buffers(msj)
    n_rows = 125_000_000                       # obs alone: 4.5 GB
    big = [torch.empty((n_rows,) + t.shape[1:], dtype=t.dtype, device=DEV) for t in small]
    src = shuffled(msj, 5000)
    dst = n_rows - 1 - torch.arange(5000, device=DEV) * 7          # rows near the end
    for b, s in zip(big, small):
        b[dst] = s[src]
    image = pack_policy_image(msj.policy)
    g1, s1 = ppo_grad(image, *small, src)
    g2, s2 = ppo_grad(image, *big, dst.contiguous())
    torch.cuda.synchronize()
    assert torch.equal(g1.view(torch.int32), g2.view(torch.int32)) and torch.equal(s1.view(torch.int64), s2.view(torch.int64))
    del big


def test_first_minibatch_after_an_fp32_collect():
    col = collected(None)
    _, s, _ = kernel(col.policy, buffers(col), shuffled(col, 8192))
    assert s["approxkl"] < 1e-10 and s["clipfrac"] == 0.0


def test_out_of_range_indices_are_counted_and_skipped(msj):
    bufs = buffers(msj)
    idx = away_from_boundaries(msj.policy, bufs, shuffled(msj, 3000))
    bad = idx.clone()
    bad[::10] = -1
    bad[5::10] = bufs[0].shape[0] + 3
    g64, s64, _, _ = reference(msj.policy, bufs, bad)
    g32, _, _, _ = reference(msj.policy, bufs, bad, dtype=torch.float32)
    gk, sk, _ = kernel(msj.policy, bufs, bad)
    assert sk["bad_indices"] == float(((bad < 0) | (bad >= bufs[0].shape[0])).sum())
    for name in PARAMS:
        err_k, err_32 = float((gk[name] - g64[name]).abs().max()), float((g32[name] - g64[name]).abs().max())
        assert err_k <= 8 * err_32 + 2e-6 * float(g64[name].abs().max()), name
    assert abs(sk["pg_loss"] - s64["pg_loss"]) <= 1e-5 * abs(s64["pg_loss"])


def test_nan_observation_gives_nan_where_float64_does(msj):
    obs, *rest = buffers(msj)
    obs = obs.clone()
    idx = shuffled(msj, 500)
    obs[idx[17]] = float("nan")
    bufs = (obs, *rest)
    g64, _, _, _ = reference(msj.policy, bufs, idx)
    gk, _, _ = kernel(msj.policy, bufs, idx)
    for name in PARAMS:
        assert torch.equal(torch.isnan(gk[name]).cpu(), torch.isnan(g64[name]).cpu()), name


def test_refusals_are_returned():
    from gym_roboy_b200 import _native
    from gym_roboy_b200.ppo import ppo_workspace_bytes
    lib = _native.load()
    P = _native.policy_layout(9, 8)[_native.POLICY_LAYOUT_FLOATS]
    img, grad = (torch.zeros(P + 4, device=DEV) for _ in range(2))
    rows = 64
    obs, act = torch.zeros((rows, 9), device=DEV), torch.zeros((rows, 8), device=DEV)
    vec = torch.zeros(rows, device=DEV)
    idx = torch.zeros(16, dtype=torch.int64, device=DEV)
    stats = torch.zeros(9, dtype=torch.float64, device=DEV)
    need = ppo_workspace_bytes(9, 8, 16)
    ws = torch.zeros(need, dtype=torch.uint8, device=DEV)
    p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731

    def call(D=9, A=8, image=img, M=16, index=idx, o=obs, w=ws, ptr_img=None, ptr_ws=None):
        return lib.roboy_ppo_grad(D, A, ptr_img if ptr_img is not None else p(image), M, p(index), rows, p(o), p(act),
                                  p(vec), p(vec), p(vec), 0.2, 0.2, 0.01, 0.5, p(grad), p(stats),
                                  ptr_ws if ptr_ws is not None else p(w), None)
    assert call() == 0
    torch.cuda.synchronize()
    assert call(D=10) == -1 and call(D=48) == -1 and call(A=0) == -1 and call(A=65) == -1
    assert call(M=0) == -1
    assert call(index=None) == -1 and call(o=None) == -1 and call(image=None) == -1 and call(w=None) == -1
    assert call(ptr_img=ctypes.c_void_p(img.data_ptr() + 4)) == -1 and b"aligned" in lib.roboy_last_error()
    # a workspace that ends before roboy_ppo_workspace_bytes: its last bytes placed at the end of the allocation
    seg = next(s for s in torch.cuda.memory_snapshot()
               if s["address"] <= ws.data_ptr() < s["address"] + s["total_size"])
    end = seg["address"] + seg["total_size"]
    assert call(ptr_ws=ctypes.c_void_p((end - need + 8) & ~7)) == -1 and b"workspace" in lib.roboy_last_error()
    assert call(ptr_ws=ctypes.c_void_p(end - need)) == 0
    torch.cuda.synchronize()


def test_trainer_minibatches_match_the_reference():
    from gym_roboy_b200.envs import RoboyEnv
    from gym_roboy_b200.envs.simulations import CudaSimulationClient
    from gym_roboy_b200.ppo import PPO2
    from gym_roboy_b200.rollout import MlpPolicy
    torch.manual_seed(0)
    env = RoboyEnv(CudaSimulationClient(num_envs=4096, seed=9, device=DEV), strict=False)
    model = PPO2(env, MlpPolicy().to(DEV), n_steps=8, nminibatches=3, noptepochs=2, seed=4)
    seen, perms = [], []
    n_batch = 4096 * 8
    # the permutations the trainer must draw: one randperm per epoch from a generator seeded by `seed`
    expect = torch.Generator(device=DEV).manual_seed(4)

    def hook(m, idx, grad, stats):
        from gym_roboy_b200.ppo import unpack_policy_grad
        mb = len(seen) % len(m.bounds)
        if mb == 0:
            perms.append(torch.randperm(n_batch, generator=expect, device=DEV))
        s, e = m.bounds[mb]
        assert torch.equal(idx, perms[-1][s:e]), (len(perms), mb)
        bufs = m._flat_buffers()
        ref = copy.deepcopy(m.policy)
        g64, _, _, _ = reference(ref, bufs, idx)
        g32, _, _, _ = reference(ref, bufs, idx, dtype=torch.float32)
        q = copy.deepcopy(m.policy)
        unpack_policy_grad(q, grad)
        for name, t in q.named_parameters():
            err_k = float((t.grad.double() - g64[name]).abs().max())
            err_32 = float((g32[name] - g64[name]).abs().max())
            # no boundary filtering here: allow the samples float32 puts on the other side of a clip boundary
            assert err_k <= 8 * err_32 + 2e-6 * float(g64[name].abs().max()) + 1e-6, name
        seen.append(idx.numel())
    model.learn(4096 * 8, minibatch_hook=hook)
    assert seen == [10922, 10922, 10922, 2] * 2 and len(model.logs) == 1
    assert len(perms) == 2 and not torch.equal(perms[0], perms[1])


@pytest.mark.parametrize("robot,fused", [("msj", "fp32"), ("msj", "tc_exact"), ("fifteen_joints_64_tendons", "fp32")])
def test_trainer_is_reproducible(robot, fused):
    from gym_roboy_b200.envs import RoboyEnv
    from gym_roboy_b200.envs.simulations import CudaSimulationClient
    from gym_roboy_b200.ppo import PPO2
    from gym_roboy_b200.rollout import MlpPolicy
    runs = []
    for _ in range(2):
        client = CudaSimulationClient(robot=robot_from_bounds(ROBOTS[robot]), num_envs=4096, seed=2, device=DEV)
        torch.manual_seed(0)
        policy = MlpPolicy(client.dim_obs, client.dim_action).to(DEV)
        model = PPO2(RoboyEnv(client, strict=False), policy, n_steps=8, fused=fused, seed=7).learn(2 * 4096 * 8)
        runs.append([q.detach().clone() for q in policy.parameters()])
        assert len(model.logs) == 2 and all(math.isfinite(v) for v in model.logs[-1].values())
    for a, b in zip(*runs):
        assert torch.isfinite(a).all() and torch.equal(a, b)
