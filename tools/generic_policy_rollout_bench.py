"""Closed-loop rollouts of robots other than MSJ: the float32 fused rollout (`fused="fp32"`, the generic kernel) against
the torch-policy collector (`fused=False`) on the same robot, alternated in one process, with MSJ's fused kernel (K5)
as the yardstick.  T = 128.  Writes one JSON document (card name and power limit included) to stdout and to --out.

FMAs per env-step evaluated by the fused kernels: 64 * (2D + 128 + 8 + A8) with D = 3J inputs and A8 = 8 * ceil(A / 8)
policy outputs (the value network's output layer is padded to 8 columns); share of peak against the nominal FP32 rate
of the B200 (74.4 TFLOP/s, as DESIGN.md quotes for K5).

usage: python tools/generic_policy_rollout_bench.py [--envs 262144,1048576] [--rounds 2] [--out FILE]"""
import argparse
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
from gym_roboy_b200.envs import RoboyEnv  # noqa: E402
from gym_roboy_b200.envs.simulations import CudaSimulationClient  # noqa: E402
from gym_roboy_b200.rollout import MlpPolicy, RolloutCollector  # noqa: E402

T = 128
PEAK_FP32_FLOPS = 74.4e12
ROBOTS = {"msj": None, "six_joints_14_tendons": GENERIC_ROBOTS["six_joints_14_tendons"],
          "fifteen_joints_64_tendons": GENERIC_ROBOTS["fifteen_joints_64_tendons"]}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = (s.strip() for s in q.split(","))
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def time_rollouts(robot, n, fused, reps):
    torch.manual_seed(0)
    c = CudaSimulationClient(robot=robot_from_bounds(robot), num_envs=n, seed=1, device="cuda:0")
    env = RoboyEnv(c, strict=False)
    env._single = False
    policy = MlpPolicy(c.dim_obs, c.dim_action).to("cuda:0")
    col = RolloutCollector(env, policy, n_steps=T, fused=fused)
    col.collect()   # warm-up: module load, torch kernels
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        col.collect()
    e.record()
    torch.cuda.synchronize()
    ms = s.elapsed_time(e) / reps
    dims = (c.dim_obs, c.dim_action, c.msj_kernels)
    c.close()
    del col, env, c, policy
    torch.cuda.empty_cache()
    return ms, dims


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", default="262144,1048576")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    sizes = [int(x) for x in a.envs.split(",")]
    info = card()
    rows = {}
    for rnd in range(a.rounds):
        for name, robot in ROBOTS.items():
            for n in sizes:
                for fused in ("fp32", False):   # alternated: fused, torch, fused, torch ...
                    if name == "msj" and fused is False:
                        continue
                    ms, (D, A, msj) = time_rollouts(robot, n, fused, reps=3 if fused else 1)
                    mode = fused or "torch"
                    rows.setdefault((name, n, mode), []).append(ms)
                    print(name, n, mode, "round", rnd, "ms/rollout %.2f" % ms, file=sys.stderr, flush=True)
                    rows[(name, n, mode, "dims")] = (D, A, msj)
    out = dict(card=info, T=T, rounds=a.rounds, timing="CUDA events around `reps` collect() calls after one warm-up "
               "(fused: 3 reps, torch: 1), mean over rounds; collect() includes GAE and the obs hand-over", results=[])
    for (name, n, mode), ms_list in sorted((k, v) for k, v in rows.items() if len(k) == 3):
        D, A, msj = rows[(name, n, mode, "dims")]
        fused = mode == "fp32"
        ms = sum(ms_list) / len(ms_list)
        sps = n * T / ms * 1e3
        row = dict(robot=name, envs=n, fused=mode, kernel=("K5 (MSJ)" if msj else "generic") if fused else "torch policy + step",
                   ms_per_rollout=ms, ms_all_rounds=ms_list, env_steps_per_s=sps, dim_obs=D, dim_action=A)
        if fused:
            a8 = (A + 7) // 8 * 8
            fma = 64 * (2 * D + 128 + 8 + a8)
            row.update(fma_per_env_step=fma, tflops=2 * fma * sps / 1e12, share_of_fp32_peak=2 * fma * sps / PEAK_FP32_FLOPS)
            base = rows.get((name, n, "torch"))
            if base:
                row["speedup_vs_torch"] = sum(base) / len(base) / ms
        out["results"].append(row)
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
