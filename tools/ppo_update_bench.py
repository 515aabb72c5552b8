"""PPO2 update on one GPU: the minibatch-gradient kernel (roboy_ppo_grad) against torch autograd on the same minibatch,
and one full PPO2.learn update split into collect and update.

    python tools/ppo_update_bench.py --out profiles/r3_ppo_update.json

Same-minibatch comparison: float32 with TF32 off, kernel and torch alternated in one process, CUDA events around each
call (reps after a warm-up), peak device memory of each above the inputs.  Buffers of 1,048,576 rows are gathered by a
random index of M rows (with repeats), so the gathered data (> 126 MB L2 at the larger M) streams from HBM.
Share of peak: algorithmic FMAs per sample 256 D + 24,576 + 192 (A + 1), at 2 FLOP each, over the nominal 74.4 TFLOP/s
FP32 peak; bytes per sample: the index (8), obs (4 D), actions (4 A), logp / value / return (12).
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

FP32_PEAK = 74.4e12
HBM_BW = 7.7e12
# joints, tendons, angle / velocity / tendon bound (symmetric, the same for every component); None: MsjRobot
ROBOTS = {"msj": None, "six_joints_14_tendons": (6, 14, 2.5, 0.6, 0.2), "fifteen_joints_64_tendons": (15, 64, 2.0, 0.5, 0.3)}


def dims(name):
    r = ROBOTS[name]
    return (9, 8) if r is None else (3 * r[0], r[1])


def robot(name):
    """A RoboyRobot plug-in with the spaces of ROBOTS[name] (None for MSJ: the client's default robot)."""
    if ROBOTS[name] is None:
        return None
    from gym_roboy_b200.envs.robots import RoboyRobot
    from gym_roboy_b200.spaces import Box
    J, A, a, v, t = ROBOTS[name]

    class Robot(RoboyRobot):
        _A, _V, _T = Box(-a, a, (J,), "float32"), Box(-v, v, (J,), "float32"), Box(-t, t, (A,), "float32")
        get_action_space = classmethod(lambda cls: cls._T)
        get_joint_angles_space = classmethod(lambda cls: cls._A)
        get_joint_vels_space = classmethod(lambda cls: cls._V)
    return Robot()


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def fmas(D, A):
    return 256 * D + 24576 + 192 * (A + 1)


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / 1e3 / reps


def peak_above(fn, base):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


def torch_step(policy, bufs, idx, clip=0.2, ent_coef=0.01, vf_coef=0.5):
    obs, actions, logp, values, ret = bufs
    o, a, lp_old, v_old, R = (t[idx] for t in bufs)
    adv = R - v_old
    adv = (adv - adv.mean()) / (adv.std(unbiased=False) + 1e-8)
    mean, v = policy.pi(o), policy.vf(o).squeeze(-1)
    z = (a - mean) / policy.log_std.exp()
    lp = -0.5 * (z * z).sum(-1) - 0.5 * a.shape[-1] * 1.8378770664093453 - policy.log_std.sum()
    ratio = torch.exp(lp - lp_old)
    pg1, pg2 = -adv * ratio, -adv * torch.clamp(ratio, 1 - clip, 1 + clip)
    l1 = (v - R) ** 2
    l2 = (v_old + torch.clamp(v - v_old, -clip, clip) - R) ** 2
    loss = (torch.where(pg1 >= pg2, pg1, pg2).mean() - ent_coef * (policy.log_std + 1.4189385332046727).sum()
            + vf_coef * 0.5 * torch.where(l1 >= l2, l1, l2).mean())
    policy.zero_grad(set_to_none=False)
    loss.backward()


def same_minibatch(name, M, rows=1 << 20, reps=5):
    from gym_roboy_b200.ppo import ppo_grad, ppo_workspace_bytes
    from gym_roboy_b200.rollout import MlpPolicy, pack_policy_image
    D, A = dims(name)
    torch.manual_seed(0)
    dev = "cuda:0"
    policy = MlpPolicy(D, A).to(dev)
    bufs = (torch.randn(rows, D, device=dev), torch.randn(rows, A, device=dev), torch.randn(rows, device=dev) - 5.0,
            torch.randn(rows, device=dev), torch.randn(rows, device=dev))
    idx = torch.randint(0, rows, (M,), device=dev)
    image = pack_policy_image(policy)
    grad = torch.empty_like(image)
    stats = torch.empty(9, dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    ws = torch.empty(ppo_workspace_bytes(D, A, M), dtype=torch.uint8, device=dev)
    kern = lambda: ppo_grad(image, *bufs, idx, grad=grad, stats=stats, workspace=ws)  # noqa: E731
    rec = dict(robot=name, D=D, A=A, M=M, fma_per_sample=fmas(D, A), workspace_bytes=ws.numel())
    rec["kernel_peak_bytes"] = peak_above(kern, base)   # base is read before the workspace is allocated: it counts
    t_k, t_t = [], []
    torch_ok = True
    for _ in range(2):   # alternated
        t_k.append(timed(kern, reps))
        if torch_ok:
            try:
                t_t.append(timed(lambda: torch_step(policy, bufs, idx), max(1, reps // 2)))
            except torch.OutOfMemoryError:
                torch_ok = False
                torch.cuda.empty_cache()
    tk = min(t_k)
    rec.update(kernel_s=tk, kernel_samples_per_s=M / tk,
               kernel_fp32_peak_share=2 * fmas(D, A) * M / tk / FP32_PEAK,
               kernel_hbm_share=(8 + 4 * D + 4 * A + 12) * M / tk / HBM_BW)
    if torch_ok and t_t:
        tt = min(t_t)
        torch.cuda.empty_cache()
        rec.update(torch_s=tt, torch_samples_per_s=M / tt, torch_fp32_peak_share=2 * fmas(D, A) * M / tt / FP32_PEAK,
                   torch_peak_bytes=peak_above(lambda: torch_step(policy, bufs, idx), base), kernel_speedup=tt / tk)
    else:
        rec["torch"] = "out of memory"
    return rec


def one_update(name, fused, n=1 << 20, T=128):
    from gym_roboy_b200.envs import RoboyEnv
    from gym_roboy_b200.envs.simulations import CudaSimulationClient
    from gym_roboy_b200.ppo import PPO2
    from gym_roboy_b200.rollout import MlpPolicy
    client = CudaSimulationClient(robot=robot(name), num_envs=n, seed=1, device="cuda:0")
    torch.manual_seed(0)
    model = PPO2(RoboyEnv(client, strict=False), MlpPolicy(client.dim_obs, client.dim_action).to("cuda:0"),
                 n_steps=T, fused=fused)
    col = model.collector
    orig = col.collect
    spent = []

    def collect():
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        orig()
        torch.cuda.synchronize()
        spent.append(time.perf_counter() - t0)
        return col
    col.collect = collect
    model.learn(n * T)            # warm-up update
    spent.clear()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    model.learn(n * T)
    torch.cuda.synchronize()
    total = time.perf_counter() - t0
    return dict(robot=name, fused=fused, n_envs=n, T=T, total_s=total, collect_s=spent[0], update_s=total - spent[0],
                minibatches=len(model.bounds) * model.noptepochs, logs=model.logs[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="262144,8388608,33554432")
    ap.add_argument("--skip-learn", action="store_true")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    out = dict(card=card(), same_minibatch=[], learn=[])
    for name in ROBOTS:
        for M in (int(m) for m in args.sizes.split(",")):
            r = same_minibatch(name, M)
            print(json.dumps(r), flush=True)
            out["same_minibatch"].append(r)
            torch.cuda.empty_cache()
    if not args.skip_learn:
        for name, fused in (("msj", "tc_exact"), ("fifteen_joints_64_tendons", "fp32")):
            r = one_update(name, fused)
            print(json.dumps(r), flush=True)
            out["learn"].append(r)
            torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
