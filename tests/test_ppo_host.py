"""PPO2 host logic without a GPU: schedules, minibatch partitioning, the gradient image layout, the optimizer step
against TF's formulas in float64, and the argument checks of roboy_ppo_grad / roboy_ppo_workspace_bytes."""
import ctypes
import math

import pytest
import torch

from gym_roboy_b200 import _native
from gym_roboy_b200.ppo import (TFAdam, clip_by_global_norm, minibatch_bounds, ppo_workspace_bytes, progress_fraction,
                                schedule, unpack_policy_grad)
from gym_roboy_b200.rollout import MlpPolicy, pack_policy_image


def test_schedules_and_progress_fraction():
    assert schedule(0.2)(0.3) == 0.2
    f = lambda frac: 2.5e-4 * frac  # noqa: E731
    assert schedule(f) is f
    assert [progress_fraction(u, 4) for u in (1, 2, 3, 4)] == [1.0, 0.75, 0.5, 0.25]


def test_minibatch_bounds_with_remainder():
    assert minibatch_bounds(16, 4) == [(0, 4), (4, 8), (8, 12), (12, 16)]
    assert minibatch_bounds(10, 3) == [(0, 3), (3, 6), (6, 9), (9, 10)]
    assert minibatch_bounds(5, 5) == [(i, i + 1) for i in range(5)]
    with pytest.raises(ValueError):
        minibatch_bounds(3, 4)


@pytest.mark.parametrize("dims", [(9, 8), (18, 14), (15, 11), (45, 64), (3, 1)])
def test_unpack_inverts_pack(dims):
    torch.manual_seed(0)
    pol = MlpPolicy(*dims)
    with torch.no_grad():
        pol.log_std.normal_()
    img = pack_policy_image(pol)
    s = _native.policy_layout(*dims)[_native.POLICY_LAYOUT_STD]
    img[s: s + dims[1]] = pol.log_std.detach()       # a gradient image carries d/d log_std in the std slots
    q = MlpPolicy(*dims)
    unpack_policy_grad(q, img)
    for (name, a), b in zip(pol.named_parameters(), q.parameters()):
        assert b.grad.shape == a.shape and torch.equal(b.grad, a.detach()), name


def test_clip_and_adam_equal_tf_formulas_in_float64():
    torch.manual_seed(1)
    params = [torch.nn.Parameter(torch.randn(5, 3)), torch.nn.Parameter(torch.randn(7))]
    opt = TFAdam(params)
    p64 = [p.detach().double().clone() for p in params]
    m64 = [torch.zeros_like(p) for p in p64]
    v64 = [torch.zeros_like(p) for p in p64]
    for t in range(1, 4):
        grads = [torch.randn_like(p) * 3 for p in params]
        for p, g in zip(params, grads):
            p.grad = g.clone()
        clip_by_global_norm([p.grad for p in params], 0.5)
        opt.step(2.5e-4)
        g64 = [g.double() for g in grads]
        norm = math.sqrt(sum(float((g * g).sum()) for g in g64))
        g64 = [g * 0.5 / max(norm, 0.5) for g in g64]
        lr_t = 2.5e-4 * math.sqrt(1 - 0.999 ** t) / (1 - 0.9 ** t)
        for i, g in enumerate(g64):
            m64[i] = 0.9 * m64[i] + 0.1 * g
            v64[i] = 0.999 * v64[i] + 0.001 * g * g
            p64[i] = p64[i] - lr_t * m64[i] / (v64[i].sqrt() + 1e-5)
        for p, r in zip(params, p64):
            assert float(((p.detach().double() - r).abs() / r.abs()).max()) <= 1e-6


def test_argument_checks_without_a_gpu():
    lib = _native.load()
    out = ctypes.c_uint64()
    assert lib.roboy_ppo_workspace_bytes(9, 8, 0, ctypes.byref(out)) == -1
    assert lib.roboy_ppo_workspace_bytes(10, 8, 5, ctypes.byref(out)) == -1
    assert lib.roboy_ppo_workspace_bytes(9, 65, 5, ctypes.byref(out)) == -1
    assert lib.roboy_ppo_workspace_bytes(9, 8, 5, None) == -1
    # one 64-sample tile: 256 CTA partials of (sum, sum of squares, bad), one slot's 4 loss sums and its gradient image
    P = _native.policy_layout(9, 8)[_native.POLICY_LAYOUT_FLOATS]
    assert ppo_workspace_bytes(9, 8, 5) == 8 * (3 * 256 + 4) + 4 * P
    assert ppo_workspace_bytes(45, 64, 1 << 30) == 8 * (3 * 256 + 4 * 1184) + 4 * 1184 * _native.policy_layout(45, 64)[
        _native.POLICY_LAYOUT_FLOATS]
    args = [9, 8, None, 16, None, 64] + [None] * 5 + [0.2, 0.2, 0.01, 0.5] + [None] * 4
    assert lib.roboy_ppo_grad(*args) == -1 and b"NULL" in lib.roboy_last_error()
    args[3] = 0
    assert lib.roboy_ppo_grad(*args) == -1 and b"M == 0" in lib.roboy_last_error()
    args[0], args[3] = 10, 16
    assert lib.roboy_ppo_grad(*args) == -1 and b"dim_obs" in lib.roboy_last_error()
