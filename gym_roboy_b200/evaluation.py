"""Deterministic policy evaluation on the GPU: stable-baselines' `evaluate_policy(model, env, n_eval_episodes,
deterministic=True)` for a batched `RoboyEnv`, in one kernel launch.

`evaluate_policy` plays the policy mean `clip(pi(obs), -1, 1)` in every env for exactly `n_steps` steps inside the
env kernel (`roboy_policy_evaluate`): no per-step launch, no `[T, N]` buffer.  Each env records its first
`n_eval_episodes` episodes that start inside the call -- return (the float64 sum of the float32 step rewards, in step
order, as stable-baselines sums them), length and whether the goal was reached -- and counts every such episode that
finished.  An episode already in progress when the call starts is not counted.
"""
import ctypes
from dataclasses import dataclass

import torch

from . import _native
from .rollout import pack_policy_image


@dataclass
class EvaluationResult:
    """Per-episode records `[K, N]` (slot `[k, e]`: the k-th counted episode of env e; unfilled slots hold NaN, 0,
    False), `completed` `[N]` (every counted episode that finished, beyond K too), and the summary over the recorded
    episodes: `mean_return` / `std_return` (stable-baselines' pair; population std), `success_rate` (share of recorded
    episodes that reached the goal) and `mean_length`."""
    returns: torch.Tensor     # float64 [K, N]
    lengths: torch.Tensor     # int32 (uint32 values) [K, N]
    reached: torch.Tensor     # bool [K, N]
    completed: torch.Tensor   # int32 (uint32 values) [N]
    n_steps: int
    mean_return: float
    std_return: float
    success_rate: float
    mean_length: float

    @property
    def n_episodes(self):
        """Number of recorded episodes."""
        return int((~torch.isnan(self.returns)).sum().item())


def default_n_steps(max_episode_len, n_eval_episodes, reset=True):
    """The smallest step count that guarantees `n_eval_episodes` complete counted episodes in every env.

    An episode ends at the latest when its step counter passes `max_episode_len` (roboy_env.py:72-73): a counter starts
    at 1 on reset and grows by one per step, so an episode that starts inside the call lasts at most L =
    max(max_episode_len, 1) steps.  After a reset every env starts a counted episode at the first step: K * L steps.
    Without one, an env may be in the middle of an episode that is not counted; it ends within L steps, so one L more."""
    L = max(int(max_episode_len), 1)
    return (int(n_eval_episodes) + (0 if reset else 1)) * L


@torch.no_grad()
def evaluate_policy(env, policy, n_eval_episodes=1, n_steps=None, reset=True):
    """Play `policy` (an `MlpPolicy(3J, A)` of the env's robot) deterministically in every env of `env` and record
    the first `n_eval_episodes` episodes of each env that start inside the call.

    `reset=True` resets every env first.  `n_steps=None` takes `default_n_steps`, enough for `n_eval_episodes` complete
    episodes per env.  The env needs auto-reset on.  The env continues from where the evaluation left it: its
    observation buffer holds the observation after the last step, and the call counter, goals, step counters, error word
    and episode statistics have advanced as for `n_steps` calls of `env.step`."""
    client = env._simulation_client
    dev, n = client.device, client.num_envs
    K = int(n_eval_episodes)
    if K < 0:
        raise ValueError("n_eval_episodes must be >= 0")
    T = default_n_steps(client._cfg.max_episode_len, K, reset) if n_steps is None else int(n_steps)
    if not 0 <= T < 2 ** 32:
        raise ValueError("n_steps must be in [0, 2^32)")
    # an image of the robot's dims: a policy of other dims fails in pack_policy_image
    image = torch.zeros(_native.policy_layout(client.dim_obs, client.dim_action)[_native.POLICY_LAYOUT_FLOATS],
                        dtype=torch.float32, device=dev)
    pack_policy_image(policy, out=image)
    if reset:
        env.reset()
    # allocated with one row at least: K = 0 still hands the library valid pointers (an empty view has none)
    bufs = [torch.empty((max(K, 1), n), dtype=dt, device=dev) for dt in (torch.float64, torch.int32, torch.uint8)]
    completed = torch.empty((n,), dtype=torch.int32, device=dev)
    if T == 0:   # the call launches nothing: nothing was played
        bufs[0].fill_(float("nan")); bufs[1].zero_(); bufs[2].zero_(); completed.zero_()
    p = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    _native.check(_native.load().roboy_policy_evaluate(client._h, T, p(image), p(client.obs), K, *(p(b) for b in bufs),
                                                       p(completed), stream))
    returns, lengths, reached = (b[:K] for b in bufs)
    rec = ~torch.isnan(returns)
    m = int(rec.sum().item())
    r = returns[rec]
    nan = float("nan")
    return EvaluationResult(
        returns=returns, lengths=lengths, reached=reached.view(torch.bool), completed=completed, n_steps=T,
        mean_return=float(r.mean().item()) if m else nan,
        std_return=float(r.std(unbiased=False).item()) if m else nan,
        success_rate=float(reached[rec].double().mean().item()) if m else nan,
        mean_length=float(lengths[rec].double().mean().item()) if m else nan)
