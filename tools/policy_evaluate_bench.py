"""Deterministic policy evaluation, three ways, on the same robot and population size, alternated in one process:
  * "evaluate": the fused evaluator (`roboy_policy_evaluate`, one launch for T steps, per-episode records only);
  * "torch": a torch loop over the env step -- policy.pi(obs), clamp, env step, per-episode bookkeeping in torch
    (float64 running return, records written on done) -- what a user without the evaluator writes;
  * "rollout_std0": `RolloutCollector(fused="fp32")` with log_std = -200 (std exactly 0), which stores [T+1, N, ...]
    buffers; skipped where they do not fit in --mem-cap GB.
T = 400 (one MSJ episode), K = 1 record per env.  Writes one JSON document (card name and power limit included) to
stdout and to --out.

FMAs per env-step evaluated by the evaluator: 64 * (D + 64 + A8), D = 3J inputs, A8 = 8 * ceil(A / 8) policy outputs;
share of peak against the nominal FP32 rate of the B200 (74.4 TFLOP/s, as tools/generic_policy_rollout_bench.py).

usage: python tools/policy_evaluate_bench.py [--envs 262144,1048576] [--rounds 2] [--out FILE]"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402

from cuda_adaptor import robot_from_bounds  # noqa: E402
from test_oracle_vs_reference import GENERIC_ROBOTS  # noqa: E402
from gym_roboy_b200 import _native  # noqa: E402
from gym_roboy_b200.envs import RoboyEnv  # noqa: E402
from gym_roboy_b200.envs.simulations import CudaSimulationClient  # noqa: E402
from gym_roboy_b200.rollout import MlpPolicy, RolloutCollector, pack_policy_image  # noqa: E402

T = 400
K = 1
PEAK_FP32_FLOPS = 74.4e12
ROBOTS = {"msj": None, "six_joints_14_tendons": GENERIC_ROBOTS["six_joints_14_tendons"],
          "fifteen_joints_64_tendons": GENERIC_ROBOTS["fifteen_joints_64_tendons"]}
MODES = ("evaluate", "torch", "rollout_std0")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = (s.strip() for s in q.split(","))
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def rollout_bytes(n, D, A):
    """The [T+1, N, ...] buffers of RolloutCollector: obs, actions, logp, values, rewards, dones, adv, ret."""
    return 4 * ((T + 1) * n * D + T * n * A + 5 * T * n + (T + 1) * n) + T * n


def setup(robot, n):
    torch.manual_seed(0)
    c = CudaSimulationClient(robot=robot_from_bounds(robot), num_envs=n, seed=1, device="cuda:0")
    env = RoboyEnv(c, strict=False)
    env._single = False
    policy = MlpPolicy(c.dim_obs, c.dim_action).to("cuda:0")
    return c, env, policy


def run_evaluate(c, env, policy):
    n = c.num_envs
    img = torch.zeros(_native.policy_layout(c.dim_obs, c.dim_action)[_native.POLICY_LAYOUT_FLOATS], device="cuda:0")
    pack_policy_image(policy, out=img)
    rec = [torch.empty((K, n), dtype=dt, device="cuda:0") for dt in (torch.float64, torch.int32, torch.uint8)]
    completed = torch.empty(n, dtype=torch.int32, device="cuda:0")
    p = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
    lib = _native.load()

    def once(steps):
        _native.check(lib.roboy_policy_evaluate(c._h, steps, p(img), p(c.obs), K, *(p(r) for r in rec), p(completed),
                                                ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    once(8)   # warm-up: module load
    return lambda: once(T)


def run_torch(c, env, policy):
    n = c.num_envs
    ret = torch.zeros(n, dtype=torch.float64, device="cuda:0")
    counting = torch.zeros(n, dtype=torch.bool, device="cuda:0")
    n_rec = torch.zeros(n, dtype=torch.int64, device="cuda:0")
    returns = torch.full((K, n), float("nan"), dtype=torch.float64, device="cuda:0")
    ar = torch.arange(n, device="cuda:0")
    flat = returns.view(-1)
    clipped = torch.empty((n, c.dim_action), device="cuda:0")

    def loop(steps):
        with torch.no_grad():
            counting.copy_((c.step_flags & _native.STEP_MASK) == 1)
            for _ in range(steps):
                torch.clamp(policy.pi(c.obs), -1.0, 1.0, out=clipped)
                c.step_fused(clipped)
                ret.add_(torch.where(counting, c.reward.double(), 0.0))
                fin = counting & c.done
                w = fin & (n_rec < K)
                idx = n_rec.clamp(max=K - 1) * n + ar
                flat.index_copy_(0, idx, torch.where(w, ret, flat[idx]))   # no host sync: every env writes its slot
                n_rec.add_(fin.long())
                counting.logical_or_(c.done)
                ret.masked_fill_(c.done, 0.0)
    loop(2)   # warm-up: torch kernels
    return lambda: loop(T)


def run_rollout(c, env, policy):
    with torch.no_grad():
        policy.log_std.fill_(-200.0)
    col = RolloutCollector(env, policy, n_steps=T, fused="fp32")
    col.collect()   # warm-up
    return col.collect


def time_mode(robot, n, mode, reps):
    c, env, policy = setup(robot, n)
    fn = dict(evaluate=run_evaluate, torch=run_torch, rollout_std0=run_rollout)[mode](c, env, policy)
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    torch.cuda.synchronize()
    ms = s.elapsed_time(e) / reps
    dims = (c.dim_obs, c.dim_action)
    c.close()
    del fn, env, c, policy
    torch.cuda.empty_cache()
    return ms, dims


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", default="262144,1048576")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--mem-cap", type=float, default=120.0, help="GB the std-0 rollout's buffers may take")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    sizes = [int(x) for x in a.envs.split(",")]
    info = card()
    rows, dims = {}, {}
    for rnd in range(a.rounds):
        for name, robot in ROBOTS.items():
            for n in sizes:
                for mode in MODES:   # alternated: evaluate, torch, rollout, evaluate, ...
                    D = 3 * (3 if robot is None else robot.get("dim_joint", 3))
                    A = 8 if robot is None else robot.get("dim_action", 8)
                    if mode == "rollout_std0" and rollout_bytes(n, D, A) > a.mem_cap * 1e9:
                        rows[(name, n, mode)] = None
                        continue
                    ms, dims[(name, n)] = time_mode(robot, n, mode, reps=3 if mode == "evaluate" else 1)
                    rows.setdefault((name, n, mode), []).append(ms)
                    print(name, n, mode, "round", rnd, "ms %.2f" % ms, file=sys.stderr, flush=True)
    out = dict(card=info, T=T, episodes=K, rounds=a.rounds,
               timing="CUDA events around `reps` calls after one warm-up (evaluate: 3 reps, others: 1), mean over "
                      "rounds; the three modes alternate inside each round", results=[])
    for (name, n, mode), ms_list in sorted(rows.items()):
        D, A = dims[(name, n)]
        row = dict(robot=name, envs=n, mode=mode, dim_obs=D, dim_action=A)
        if ms_list is None:
            row.update(skipped="[T+1, N, ...] buffers of %.1f GB exceed --mem-cap" % (rollout_bytes(n, D, A) / 1e9))
            out["results"].append(row)
            continue
        ms = sum(ms_list) / len(ms_list)
        sps = n * T / ms * 1e3
        row.update(ms_per_call=ms, ms_all_rounds=ms_list, env_steps_per_s=sps)
        if mode == "evaluate":
            a8 = (A + 7) // 8 * 8
            fma = 64 * (D + 64 + a8)
            row.update(fma_per_env_step=fma, tflops=2 * fma * sps / 1e12, share_of_fp32_peak=2 * fma * sps / PEAK_FP32_FLOPS)
            for other in ("torch", "rollout_std0"):
                base = rows.get((name, n, other))
                if base:
                    row["speedup_vs_" + other] = sum(base) / len(base) / ms
        out["results"].append(row)
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
