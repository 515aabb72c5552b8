"""PPO-style rollout collection on the GPU -- the caller of the env hot path.

The reference trains with stable-baselines' PPO2 over a `SubprocVecEnv`
(gym_roboy/train_parallel.py:28-35): per step the policy runs in the trainer process, the clipped
action crosses a pipe to each env process and the observation comes back the same way.  Here the
whole loop stays on one device: a torch policy reads the observation tensor the step kernel wrote,
actions are clipped on the device, and the step kernel writes observation / reward / done
straight into the `[T, N]` rollout buffers (its output pointers ARE the buffer slots).
Advantages come from the `roboy_gae` kernel.  With `fused=True` the policy itself runs inside the
env kernel (`roboy_policy_rollout`: both networks, the Gaussian sample, the clip and the env step for
all T steps in ONE launch, state in registers), which removes every per-step launch and every
activation round trip through HBM.  Because the env's call counter is device state, the
entire T-step loop can be captured in one CUDA graph and replayed, which is what makes small
populations (e.g. 4,096 envs), otherwise launch-bound, run at speed.

stable-baselines itself is not part of the reference repo (SURVEY.md 8c: parity unpinned); the
policy shape and the GAE recurrence follow its PPO2 `MlpPolicy` / runner as documented upstream:
separate 64-64 tanh networks for policy and value, state-independent log-std, actions clipped to
the action space before `env.step`.
"""
import ctypes
import math

import torch

from . import _native


class MlpPolicy(torch.nn.Module):
    def __init__(self, obs_dim=9, act_dim=8, hidden=64):
        super().__init__()
        def net(out):
            return torch.nn.Sequential(torch.nn.Linear(obs_dim, hidden), torch.nn.Tanh(),
                                       torch.nn.Linear(hidden, hidden), torch.nn.Tanh(), torch.nn.Linear(hidden, out))
        self.pi, self.vf = net(act_dim), net(1)
        self.log_std = torch.nn.Parameter(torch.zeros(act_dim))

    def forward(self, obs):
        return self.pi(obs), self.vf(obs).squeeze(-1)


def gae(rewards, values, dones, last_value, gamma=0.99, lam=0.95, adv=None, ret=None):
    """GAE(lambda) on the device via the `roboy_gae` kernel.  rewards/values float32 [T,N], dones
    uint8/bool [T,N] (done[t]: the episode ended at step t), last_value float32 [N]."""
    T, n = rewards.shape
    adv = torch.empty_like(rewards) if adv is None else adv
    ret = torch.empty_like(rewards) if ret is None else ret
    d = dones.view(torch.uint8) if dones.dtype == torch.bool else dones
    for t in (rewards, values, d, last_value, adv, ret):
        assert t.is_cuda and t.is_contiguous()
    p = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
    stream = ctypes.c_void_p(torch.cuda.current_stream(rewards.device).cuda_stream)
    _native.check(_native.load().roboy_gae(T, n, p(rewards), p(values), p(d), p(last_value), float(gamma), float(lam),
                                           p(adv), p(ret), stream))
    return adv, ret


def pack_policy_image(policy, out=None):
    """Pack an `MlpPolicy(obs_dim=3J, act_dim=A)` into the float32 image `roboy_policy_rollout` reads, at the offsets
    `roboy_policy_layout` gives (include/roboy_b200.h): per network W1^T | b1 | W2^T | b2 | W3^T | b3 with the output
    columns zero-padded to 8 (value) or to a multiple of 8 (policy), value network first, then std = exp(log_std)
    and the log-density constant.  For MSJ (9, 8) that is the ROBOY_POLICY_OFF_* image."""
    N = _native
    dev = policy.log_std.device
    l1 = policy.pi[0]
    d_obs, d_act = l1.weight.shape[1], policy.log_std.numel()
    off = N.policy_layout(d_obs, d_act)
    a8 = (d_act + 7) // 8 * 8
    H = N.POLICY_HIDDEN
    img = torch.zeros(off[N.POLICY_LAYOUT_FLOATS], dtype=torch.float32, device=dev) if out is None else out
    assert img.numel() == off[N.POLICY_LAYOUT_FLOATS] and img.dtype == torch.float32
    for base, net, n_out, cols, b3_at in ((off[N.POLICY_LAYOUT_VF], policy.vf, 1, 8, off[N.POLICY_LAYOUT_VF_B3]),
                                          (off[N.POLICY_LAYOUT_PI], policy.pi, d_act, a8, off[N.POLICY_LAYOUT_PI_B3])):
        l1, l2, l3 = net[0], net[2], net[4]
        assert l1.weight.shape == (H, d_obs) and l2.weight.shape == (H, H) and l3.weight.shape == (n_out, H)
        w1, b1, w2, b2, w3 = (base + off[k] for k in (N.POLICY_LAYOUT_W1, N.POLICY_LAYOUT_B1, N.POLICY_LAYOUT_W2,
                                                       N.POLICY_LAYOUT_B2, N.POLICY_LAYOUT_W3))
        b3 = base + b3_at
        img[w1:b1].copy_(l1.weight.detach().t().reshape(-1))
        img[b1:w2].copy_(l1.bias.detach())
        img[w2:b2].copy_(l2.weight.detach().t().reshape(-1))
        img[b2:w3].copy_(l2.bias.detach())
        w3v = img[w3:b3].view(H, cols)
        w3v.zero_()
        w3v[:, :n_out].copy_(l3.weight.detach().t())
        b3v = img[b3:b3 + cols]
        b3v.zero_()
        b3v[:n_out].copy_(l3.bias.detach())
    log_std = policy.log_std.detach()
    std = img[off[N.POLICY_LAYOUT_STD]: off[N.POLICY_LAYOUT_LOGNORM]]
    std.zero_()
    std[:d_act].copy_(log_std.exp())
    img[off[N.POLICY_LAYOUT_LOGNORM]:].zero_()
    img[off[N.POLICY_LAYOUT_LOGNORM]] = -0.5 * math.log(2 * math.pi) * log_std.numel() - log_std.sum()
    return img


def _umma_k_major_f16(w, bias, n_pad, k_pad, bias_col):
    """[out, in] weight (+ bias as input column `bias_col`) -> zero-padded [n_pad, k_pad] split into float16 halves
    (hi = float16(w), lo = float16(w - hi)), each in the tensor core's K-major core-matrix layout without swizzle:
    element index of W[n][k] = (n//8)*(k_pad//8)*64 + (k//8)*64 + (n%8)*8 + (k%8).  Returns (hi, lo), flat."""
    full = torch.zeros((n_pad, k_pad), dtype=torch.float32, device=w.device)
    full[: w.shape[0], : w.shape[1]] = w.detach().float()
    full[: w.shape[0], bias_col] = bias.detach().float()
    hi = full.to(torch.float16)
    lo = (full - hi.float()).to(torch.float16)
    # [n/8, 8, k/8, 8] -> [n/8, k/8, 8, 8]
    lay = lambda t: t.view(n_pad // 8, 8, k_pad // 8, 8).permute(0, 2, 1, 3).reshape(-1)  # noqa: E731
    return lay(hi), lay(lo)


def pack_policy_image_tc(policy, out=None):
    """Pack an `MlpPolicy` into the byte image `roboy_policy_rollout_tc` reads (layout: ROBOY_TC_* in
    include/roboy_b200.h): float16 weights (high halves, then low halves) with the biases as an extra input column,
    then std / lognorm as float32."""
    N = _native
    dev = policy.log_std.device
    img = torch.zeros(N.TC_IMAGE_BYTES, dtype=torch.uint8, device=dev) if out is None else out
    his = img[: N.TC_OFF_LO_BYTES].view(torch.float16)
    los = img[N.TC_OFF_LO_BYTES: N.TC_OFF_STD_BYTES].view(torch.float16)
    for base, net in ((N.TC_OFF_VF, policy.vf), (N.TC_OFF_PI, policy.pi)):
        l1, l2, l3 = net[0], net[2], net[4]
        assert l1.weight.shape == (64, N.DIM_OBS) and l2.weight.shape == (64, 64) and l3.weight.shape[0] in (1, 8)
        for (lo_, hi_), layer, n_pad, k_pad, bias_col in (
                ((N.TC_OFF_W1, N.TC_OFF_W2), l1, 64, 16, N.DIM_OBS), ((N.TC_OFF_W2, N.TC_OFF_W3), l2, 64, N.TC_K_HIDDEN, 64),
                ((N.TC_OFF_W3, N.TC_NET_HALVES), l3, 16, N.TC_K_HIDDEN, 64)):
            hi, lo = _umma_k_major_f16(layer.weight, layer.bias, n_pad, k_pad, bias_col)
            his[base + lo_: base + hi_].copy_(hi)
            los[base + lo_: base + hi_].copy_(lo)
    tail = img[N.TC_OFF_STD_BYTES: N.TC_IMAGE_BYTES].view(torch.float32)
    log_std = policy.log_std.detach()
    tail[:8].copy_(log_std.exp())
    tail[8] = -0.5 * math.log(2 * math.pi) * log_std.numel() - log_std.sum()
    for i, net in enumerate((policy.vf, policy.pi)):    # float32 biases of the 64-input layers (exact mode's epilogue)
        b = tail[12 + i * N.TC_BIAS32_NET_FLOATS: 12 + (i + 1) * N.TC_BIAS32_NET_FLOATS]
        b.zero_()
        b[:64].copy_(net[2].bias.detach())
        b[64: 64 + net[4].bias.shape[0]].copy_(net[4].bias.detach())
    return img


class RolloutCollector:
    """Collects `[T, N]` rollouts from a batched `RoboyEnv` with a torch policy, all on the device.

    `actions` holds the UN-clipped Gaussian samples and `logp` their log-density (what PPO2's runner stores);
    the env is stepped with `clip(actions, -1, 1)`.  `fused="fp32"` runs policy + env for all T steps
    in one kernel launch (`roboy_policy_rollout`, float32 FFMA2 -- agrees with the torch policy to ~1e-6), on every robot;
    `fused="tc"` does the same with the matrix products on the tensor cores (`roboy_policy_rollout_tc`,
    tcgen05 with float16 operands and float32 accumulation -- agrees to ~1e-3, several times faster);
    `fused="tc_exact"` splits every operand into two float16 halves (three MMAs per product) and keeps the accurate
    tanh -- agrees to ~1e-6 like "fp32", at more than twice its speed; `fused=True` selects it.  The tensor-core variants
    run on MSJ-shaped robots only.  (`logp` is always the density of the stored
    sample under the mean the kernel computed; with "tc" that mean differs from the float32 policy's by ~1e-3, so a
    PPO ratio evaluated in float32 starts within ~1e-3 * |z| / std of 1 -- use "tc_exact" or "fp32" where that matters.)  Fused, the Gaussian noise comes from Philox keyed by
    `noise_seed` instead of torch's generator."""

    def __init__(self, env, policy, n_steps=128, gamma=0.99, lam=0.95, fused=False, noise_seed=0, envs_per_thread=0):
        self.env, self.client, self.policy = env, env._simulation_client, policy
        self.T, self.N = int(n_steps), env.num_envs
        self.gamma, self.lam = gamma, lam
        if fused not in (False, True, "fp32", "tc", "tc_exact"):
            raise ValueError('fused must be False, True / "fp32", "tc" or "tc_exact"')
        # True selects the tensor-core kernel with split float16 operands: the same ~1e-6 agreement with the float32
        # policy as the FFMA2 kernel ("fp32") at 2.8x its speed
        self.fused = {True: "tc_exact", False: None}.get(fused, fused)
        self.noise_seed, self.envs_per_thread = int(noise_seed), int(envs_per_thread)
        dev, T, N = self.client.device, self.T, self.N
        f32 = dict(dtype=torch.float32, device=dev)
        d_obs, d_act = self.client.dim_obs, self.client.dim_action
        if self.fused in ("tc", "tc_exact") and not self.client.msj_kernels:
            raise ValueError('the tensor-core policy rollouts (fused=True, "tc", "tc_exact") are built for MSJ-shaped robots; '
                             'use fused="fp32" for this robot')
        self.obs = torch.zeros((T + 1, N, d_obs), **f32)
        self.actions = torch.zeros((T, N, d_act), **f32)
        self.logp = torch.zeros((T, N), **f32)
        self.values = torch.zeros((T + 1, N), **f32)
        self.rewards = torch.zeros((T, N), **f32)
        self.dones = torch.zeros((T, N), dtype=torch.uint8, device=dev)
        self.adv = torch.zeros((T, N), **f32)
        self.ret = torch.zeros((T, N), **f32)
        self._graph = None
        self._clipped = torch.zeros((N, d_act), **f32)
        self._image, self._image_key = None, None
        if self.fused == "fp32":
            self._image = torch.zeros(_native.policy_layout(d_obs, d_act)[_native.POLICY_LAYOUT_FLOATS], **f32)
        elif self.fused in ("tc", "tc_exact"):
            self._image = torch.zeros(_native.TC_IMAGE_BYTES, dtype=torch.uint8, device=dev)
        self.noise = None   # tests: set to a [T, N, A] float32 tensor to have the fused kernel record its noise
        self.obs[0].copy_(env.reset())

    def _fused_loop(self):
        p = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
        dev = self.client.device
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        bufs = (p(self.obs), p(self.actions), p(self.logp), p(self.values), p(self.rewards), p(self.dones),
                p(self.noise) if self.noise is not None else None)
        # re-pack the weights only when a parameter changed (in-place updates bump torch's version counters);
        # inside a CUDA-graph capture the packing is always recorded, so that replays pick up new weights
        key = tuple((q.data_ptr(), q._version) for q in self.policy.parameters())
        if key != self._image_key or torch.cuda.is_current_stream_capturing():
            (pack_policy_image if self.fused == "fp32" else pack_policy_image_tc)(self.policy, out=self._image)
            self._image_key = None if torch.cuda.is_current_stream_capturing() else key
        if self.fused != "fp32":
            _native.check(_native.load().roboy_policy_rollout_tc(self.client._h, self.T, p(self._image), self.noise_seed,
                                                                 *bufs, self.envs_per_thread, int(self.fused == "tc_exact"),
                                                                 stream))
        else:
            _native.check(_native.load().roboy_policy_rollout(self.client._h, self.T, p(self._image), self.noise_seed,
                                                              *bufs, self.envs_per_thread, stream))
        gae(self.rewards, self.values[: self.T], self.dones, self.values[self.T], self.gamma, self.lam, self.adv, self.ret)
        self.obs[0].copy_(self.obs[self.T])

    def _loop(self):
        if self.fused:
            return self._fused_loop()
        policy, client = self.policy, self.client
        std = policy.log_std.exp()
        log_norm = -0.5 * math.log(2 * math.pi) * std.numel() - policy.log_std.sum()
        for t in range(self.T):
            mean, value = policy(self.obs[t])
            noise = torch.randn_like(mean)
            self.logp[t] = log_norm - 0.5 * (noise * noise).sum(-1)
            torch.addcmul(mean, std, noise, out=self.actions[t])
            torch.clamp(self.actions[t], -1.0, 1.0, out=self._clipped)        # the runner's np.clip, on the device
            self.values[t] = value
            # zero-copy: the step kernel's output pointers are the rollout buffer slots
            client.step_fused(self._clipped, obs=self.obs[t + 1], reward=self.rewards[t], done=self.dones[t])
        self.values[self.T] = policy(self.obs[self.T])[1]
        gae(self.rewards, self.values[: self.T], self.dones, self.values[self.T], self.gamma, self.lam, self.adv, self.ret)
        self.obs[0].copy_(self.obs[self.T])   # next rollout continues where this one stopped

    def state_dict(self):
        """Env checkpoint + the observation the next rollout starts from (`obs[0]`): a resumed collector continues the
        uninterrupted trajectory exactly."""
        return dict(env=self.client.state_dict(), obs0=self.obs[0].clone(), noise_seed=self.noise_seed)

    def load_state_dict(self, sd):
        self.client.load_state_dict(sd["env"])
        self.obs[0].copy_(sd["obs0"])
        self.noise_seed = int(sd["noise_seed"])

    @torch.no_grad()
    def collect(self):
        """One rollout of T steps (replays the captured CUDA graph if `capture()` was called)."""
        if self._graph is not None:
            self._graph.replay()
        else:
            self._loop()
        return self

    @torch.no_grad()
    def capture(self, warmup=1):
        """Capture the whole T-step loop (policy, clip, env step, GAE) in one CUDA graph."""
        side = torch.cuda.Stream(device=self.client.device)
        side.wait_stream(torch.cuda.current_stream(self.client.device))
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self._loop()
        torch.cuda.current_stream(self.client.device).wait_stream(side)
        torch.cuda.synchronize(self.client.device)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            self._loop()
        self._graph = graph
        return self
