"""PPO2 training on the GPU: stable-baselines 2's `PPO2` (as documented upstream) over the fused rollouts.

The update's hot path is one native call per minibatch (`roboy_ppo_grad`, gym_roboy_b200/csrc/roboy_ppo.cu): it gathers
the minibatch from the collector's `[T, N]` buffers by index, evaluates the clipped-surrogate loss and returns the
gradient of every `MlpPolicy` parameter in the layout of the packed policy image, with the loss statistics.  The
activations never leave the chip, so the memory an update needs is the rollout buffers plus a workspace of a few MB per
minibatch.  What follows the gradient -- TF's `clip_by_global_norm` and TF's Adam step -- is a handful of elementwise
torch operations on the parameters.
"""
import ctypes
import math

import torch

from . import _native
from .rollout import RolloutCollector, pack_policy_image


def _image_floats(d_obs, d_act):
    return _native.policy_layout(d_obs, d_act)[_native.POLICY_LAYOUT_FLOATS]


def ppo_workspace_bytes(d_obs, d_act, m):
    """Bytes of device workspace `roboy_ppo_grad` needs for a minibatch of m samples of this robot."""
    out = ctypes.c_uint64()
    _native.check(_native.load().roboy_ppo_workspace_bytes(int(d_obs), int(d_act), int(m), ctypes.byref(out)))
    return out.value


def ppo_grad(image, obs, actions, logp, values, ret, index, clip_range=0.2, clip_range_vf=None, ent_coef=0.01,
             vf_coef=0.5, grad=None, stats=None, workspace=None):
    """The PPO2 loss of the minibatch `index` (int64 [M], rows of the flattened buffers) and its gradient.

    `image` is the packed policy (`pack_policy_image`); `obs` [R, D], `actions` [R, A], `logp`, `values`, `ret` [R] are
    float32 device tensors (views of the collector's buffers flattened to R = T * N rows).  `clip_range_vf=None` clips
    the value with `clip_range` (stable-baselines' legacy default), a negative value turns value clipping off.
    Returns `(grad, stats)`: the gradient in the image's layout (float32 [P]) and the float64 statistics
    [`_native.PPO_STAT_NAMES`], both on the device; nothing is synchronised."""
    R, D = obs.shape
    A = actions.shape[-1]
    m = index.numel()
    dev = obs.device
    for t, shape in ((obs, (R, D)), (actions, (R, A)), (logp, (R,)), (values, (R,)), (ret, (R,))):
        if t.shape != shape or t.dtype != torch.float32 or not t.is_contiguous() or t.device != dev:
            raise ValueError("obs [R, D], actions [R, A], logp / values / ret [R]: contiguous float32 on one device")
    if index.dtype != torch.int64 or not index.is_contiguous() or index.device != dev:
        raise ValueError("index must be a contiguous int64 tensor on the buffers' device")
    if image.dtype != torch.float32 or image.numel() != _image_floats(D, A) or image.device != dev:
        raise ValueError("image must be the float32 policy image of this robot (pack_policy_image)")
    grad = torch.empty_like(image) if grad is None else grad
    stats = torch.empty(len(_native.PPO_STAT_NAMES), dtype=torch.float64, device=dev) if stats is None else stats
    need = ppo_workspace_bytes(D, A, m)
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty(need, dtype=torch.uint8, device=dev)
    cvf = float(clip_range) if clip_range_vf is None else float(clip_range_vf)
    p = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    _native.check(_native.load().roboy_ppo_grad(D, A, p(image), m, p(index), R, p(obs), p(actions), p(logp), p(values),
                                                p(ret), float(clip_range), cvf, float(ent_coef), float(vf_coef), p(grad),
                                                p(stats), p(workspace), stream))
    return grad, stats


def _layers(policy):
    """(image offset of the network, the network) for the value net and the policy net, with the layout's offsets."""
    d_obs, d_act = policy.pi[0].weight.shape[1], policy.log_std.numel()
    off = _native.policy_layout(d_obs, d_act)
    return off, ((off[_native.POLICY_LAYOUT_VF], policy.vf, 8, off[_native.POLICY_LAYOUT_VF_B3]),
                 (off[_native.POLICY_LAYOUT_PI], policy.pi, (d_act + 7) // 8 * 8, off[_native.POLICY_LAYOUT_PI_B3]))


def unpack_policy_grad(policy, grad_image):
    """The inverse of `pack_policy_image` for a gradient image: sets `.grad` of every `MlpPolicy` parameter (the std
    slots hold d loss / d log_std)."""
    N = _native
    off, nets = _layers(policy)
    H = N.POLICY_HIDDEN
    for base, net, cols, b3_at in nets:
        l1, l2, l3 = net[0], net[2], net[4]
        d_in, n_out = l1.weight.shape[1], l3.weight.shape[0]
        w1, b1, w2, b2, w3 = (base + off[k] for k in (N.POLICY_LAYOUT_W1, N.POLICY_LAYOUT_B1, N.POLICY_LAYOUT_W2,
                                                       N.POLICY_LAYOUT_B2, N.POLICY_LAYOUT_W3))
        b3 = base + b3_at
        l1.weight.grad = grad_image[w1:b1].view(d_in, H).t().contiguous()
        l1.bias.grad = grad_image[b1:w2].clone()
        l2.weight.grad = grad_image[w2:b2].view(H, H).t().contiguous()
        l2.bias.grad = grad_image[b2:w3].clone()
        l3.weight.grad = grad_image[w3:b3].view(H, cols)[:, :n_out].t().contiguous()
        l3.bias.grad = grad_image[b3:b3 + n_out].clone()
    s = off[N.POLICY_LAYOUT_STD]
    policy.log_std.grad = grad_image[s:s + policy.log_std.numel()].clone()


def schedule(value):
    """stable-baselines' `get_schedule_fn`: a constant becomes a function of the progress fraction; a callable stays."""
    return value if callable(value) else (lambda frac, v=float(value): v)


def progress_fraction(update, n_updates):
    """SB2's `frac` of update 1..n_updates: 1 at the first update, 1/n_updates at the last."""
    return 1.0 - (update - 1.0) / n_updates


def minibatch_bounds(n_batch, nminibatches):
    """SB2's minibatches over a shuffled batch: [start, end) by steps of n_batch // nminibatches, the last one holding
    the remainder when that does not divide."""
    size = n_batch // nminibatches
    if size < 1:
        raise ValueError("nminibatches must not exceed the batch (n_envs * n_steps)")
    return [(s, min(s + size, n_batch)) for s in range(0, n_batch, size)]


def clip_by_global_norm(grads, clip_norm):
    """TF's clip_by_global_norm, in place: g * c / max(||g||, c) over all tensors; returns the global norm."""
    norm = torch.sqrt(sum((g.double() * g.double()).sum() for g in grads))
    scale = (clip_norm / torch.maximum(norm, torch.tensor(float(clip_norm), dtype=torch.float64, device=norm.device)))
    for g in grads:
        g.mul_(scale.to(g.dtype))
    return norm


class TFAdam:
    """TF1's AdamOptimizer (stable-baselines' PPO2 uses epsilon = 1e-5): with t the step count,
    lr_t = lr sqrt(1 - b2^t) / (1 - b1^t);  m = b1 m + (1 - b1) g;  v = b2 v + (1 - b2) g^2;  p -= lr_t m / (sqrt(v) + eps)."""

    def __init__(self, params, beta1=0.9, beta2=0.999, eps=1e-5):
        self.params = list(params)
        self.beta1, self.beta2, self.eps = beta1, beta2, eps
        self.m = [torch.zeros_like(p) for p in self.params]
        self.v = [torch.zeros_like(p) for p in self.params]
        self.t = 0

    @torch.no_grad()
    def step(self, lr):
        self.t += 1
        lr_t = lr * math.sqrt(1.0 - self.beta2 ** self.t) / (1.0 - self.beta1 ** self.t)
        for p, m, v in zip(self.params, self.m, self.v):
            g = p.grad
            m.mul_(self.beta1).add_(g, alpha=1.0 - self.beta1)
            v.mul_(self.beta2).addcmul_(g, g, value=1.0 - self.beta2)
            p.sub_(lr_t * m / (v.sqrt() + self.eps))


class PPO2:
    """stable-baselines 2's PPO2 with its defaults, on a batched `RoboyEnv` and an `MlpPolicy` of its robot.

    Per update: one `RolloutCollector.collect()` (`fused` as there), then `noptepochs` epochs; each epoch draws a device
    `randperm` of the T * N samples from a generator seeded by `seed` and cuts it into `nminibatches` minibatches (SB2's
    trailing remainder minibatch when that does not divide).  Per minibatch: `ppo_grad`, TF's clip_by_global_norm to
    `max_grad_norm`, TF's Adam step.  `learning_rate`, `cliprange` and `cliprange_vf` take constants or functions of
    SB2's progress fraction (`progress_fraction`).  `logs` receives, per update, the means of the minibatch statistics."""

    def __init__(self, env, policy, gamma=0.99, n_steps=128, ent_coef=0.01, learning_rate=2.5e-4, vf_coef=0.5,
                 max_grad_norm=0.5, lam=0.95, nminibatches=4, noptepochs=4, cliprange=0.2, cliprange_vf=None,
                 fused="fp32", seed=0):
        if not fused:
            raise ValueError("PPO2 collects with a fused rollout: fused must be True, \"fp32\", \"tc\" or \"tc_exact\"")
        self.env, self.policy = env, policy
        self.n_steps, self.ent_coef, self.vf_coef, self.max_grad_norm = int(n_steps), ent_coef, vf_coef, max_grad_norm
        self.nminibatches, self.noptepochs = int(nminibatches), int(noptepochs)
        self.learning_rate, self.cliprange = schedule(learning_rate), schedule(cliprange)
        self.cliprange_vf = None if cliprange_vf is None else schedule(cliprange_vf)
        self.collector = RolloutCollector(env, policy, n_steps=n_steps, gamma=gamma, lam=lam, fused=fused, noise_seed=seed)
        c = self.collector
        self.device = c.client.device
        self.n_batch = c.T * c.N
        self.bounds = minibatch_bounds(self.n_batch, self.nminibatches)
        self.generator = torch.Generator(device=self.device)
        self.generator.manual_seed(int(seed))
        self.optimizer = TFAdam(policy.parameters())
        d_obs, d_act = c.client.dim_obs, c.client.dim_action
        f32 = dict(dtype=torch.float32, device=self.device)
        self._image = torch.zeros(_image_floats(d_obs, d_act), **f32)
        self._grad = torch.zeros_like(self._image)
        self._obs0 = torch.empty_like(c.obs[0])
        self._stats = torch.zeros(len(_native.PPO_STAT_NAMES), dtype=torch.float64, device=self.device)
        m_max = max(e - s for s, e in self.bounds)
        self._workspace = torch.empty(ppo_workspace_bytes(d_obs, d_act, m_max), dtype=torch.uint8, device=self.device)
        self.logs = []
        self.num_timesteps = 0

    def _flat_buffers(self):
        c = self.collector
        T, N = c.T, c.N
        return (c.obs[:T].reshape(T * N, -1), c.actions.reshape(T * N, -1), c.logp.reshape(-1),
                c.values[:T].reshape(-1), c.ret.reshape(-1))

    def learn(self, total_timesteps, minibatch_hook=None):
        """Train for total_timesteps // (n_envs * n_steps) updates.  `minibatch_hook(model, index, grad, stats)`, if
        given, is called after each minibatch's gradient, before the optimizer step."""
        n_updates = int(total_timesteps) // self.n_batch
        bufs = self._flat_buffers()
        for update in range(1, n_updates + 1):
            frac = progress_fraction(update, n_updates)
            lr, clip = self.learning_rate(frac), self.cliprange(frac)
            clip_vf = None if self.cliprange_vf is None else self.cliprange_vf(frac)
            c = self.collector
            # collect() leaves obs[0] holding the observation the NEXT rollout starts from; the update needs the one
            # this rollout started from, and the collector gets the next start back after the update
            self._obs0.copy_(c.obs[0])
            c.collect()
            c.obs[0].copy_(self._obs0)
            total = torch.zeros_like(self._stats)
            n_mb = 0
            for _ in range(self.noptepochs):
                perm = torch.randperm(self.n_batch, generator=self.generator, device=self.device)
                for s, e in self.bounds:
                    idx = perm[s:e]
                    with torch.no_grad():
                        pack_policy_image(self.policy, out=self._image)
                    ppo_grad(self._image, *bufs, idx, clip, clip_vf, self.ent_coef, self.vf_coef, grad=self._grad,
                             stats=self._stats, workspace=self._workspace)
                    if minibatch_hook is not None:
                        minibatch_hook(self, idx, self._grad, self._stats)
                    total += self._stats
                    n_mb += 1
                    self.apply_gradient(self._grad, lr)
            c.obs[0].copy_(c.obs[c.T])
            self.num_timesteps += self.n_batch
            means = (total / n_mb).tolist()
            self.logs.append(dict(zip(_native.PPO_STAT_NAMES, means), update=update, learning_rate=lr, cliprange=clip))
        return self

    def apply_gradient(self, grad_image, lr):
        """unpack_policy_grad, TF's clip_by_global_norm to max_grad_norm, TF's Adam step at learning rate lr."""
        unpack_policy_grad(self.policy, grad_image)
        if self.max_grad_norm is not None:
            clip_by_global_norm([p.grad for p in self.optimizer.params], self.max_grad_norm)
        self.optimizer.step(lr)
