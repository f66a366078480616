"""Cost of per-env physical parameters (DESIGN §5e): config C2 (two Ants, Language + tag-distance reward + distance done,
maxSteps 1024) at 4096 and 65 536 envs, step time for
  none     no parameter table (the kernels every other batch runs)
  neutral  `perEnvParams`: a table holding the model's own values (the PRM kernels, rows loaded every step)
  random   `randomizeParams` +-30 % on every family with `autoReset` and staggered episodes (resetNoise 0.05, per-env
           step counters uniform in [0, maxSteps)), so about N / 1025 envs draw new rows on every step
  auto     `autoReset` with the same staggered episodes and no table (what `random` is compared with)
Every step goes through MuJoCoRL.step with one fixed action tensor.  Timing: CUDA events on the stepping stream around
`--steps` steps after `--warmup` steps, ended by a synchronise; the L2 is not flushed.  Modes alternate within each
repeat.  Also prints the launch geometry (env-warps per CTA, shared memory per CTA) of each mode, and the GPU name and
power limit from the same run; one JSON line per measurement.

usage: python tools/bench_params.py [--envs 4096 65536] [--steps 300] [--warmup 30] [--repeats 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from mujoco_rl_environment_wrapper_b200 import plugins as P  # noqa: E402
from mujoco_rl_environment_wrapper_b200 import _lib as L  # noqa: E402
from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL  # noqa: E402

LV = os.path.join(ROOT, "tests", "levels")
MAX_STEPS = 1024
MODES = ("none", "neutral", "random", "auto")


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        out = ""
    return name, out or "unknown"


def make_env(n, mode):
    extra = {}
    if mode == "neutral":
        extra = {"perEnvParams": True}
    elif mode == "random":
        extra = {"randomizeParams": {k: [0.7, 1.3] for k in L.PARAM_FAMILIES}}
    staggered = mode in ("random", "auto")
    env = MuJoCoRL({**extra, "xmlPath": os.path.join(LV, "two_ants.xml"), "infoJson": os.path.join(LV, "info_2A.json"),
                    "agents": ["sender", "receiver"], "environmentDynamics": [P.Language],
                    "rewardFunctions": [P.tag_distance_reward], "doneFunctions": [P.distance_done], "num_envs": n,
                    "maxSteps": MAX_STEPS, "seed": 77, "autoReset": staggered, "resetNoise": 0.05 if staggered else 0.0})
    env.reset()
    if staggered:
        g = torch.Generator(device=env.device)
        g.manual_seed(5)
        env.batch.timestep.copy_(torch.randint(0, MAX_STEPS, (n,), generator=g, device=env.device, dtype=torch.int32))
    return env


def time_steps(env, steps, warmup):
    act = env.sample_actions()
    for _ in range(warmup):
        env.step(act)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        env.step(act)
    e1.record()
    torch.cuda.synchronize()
    assert torch.isfinite(env.batch.qpos).all()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, nargs="+", default=[4096, 65536])
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=30)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_params: needs a CUDA device")
    gpu, power = device_info()
    rows = []
    for n in args.envs:
        envs = {m: make_env(n, m) for m in MODES}
        times = {m: [] for m in MODES}
        for _ in range(args.repeats):
            for m in MODES:
                times[m].append(time_steps(envs[m], args.steps, args.warmup))
        for m in MODES:
            geo = envs[m].batch.geometry()
            r = {"gpu": gpu, "power_limit": power, "envs": n, "mode": m, "ms_per_step": [round(t, 5) for t in times[m]],
                 "ms_per_step_min": round(min(times[m]), 5), "warps_per_cta": geo["warps_per_cta"], "grid": geo["grid"],
                 "smem_bytes": geo["smem_bytes"]}
            rows.append(r)
            print(json.dumps(r), flush=True)
        del envs
        torch.cuda.empty_cache()
    print(f"\n{gpu}, power limit {power}; ms per step (min over {args.repeats} alternating repeats of {args.steps} steps)")
    print(f"{'envs':>6} {'mode':>8} {'ms/step':>9} {'vs none':>8} {'warps/CTA':>9} {'smem/CTA':>9}")
    for r in rows:
        base = next(x for x in rows if x["envs"] == r["envs"] and x["mode"] == "none")["ms_per_step_min"]
        print(f"{r['envs']:>6} {r['mode']:>8} {r['ms_per_step_min']:>9.4f} {r['ms_per_step_min'] / base:>8.3f} "
              f"{r['warps_per_cta']:>9} {r['smem_bytes']:>9}")
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rows, f, indent=1)


if __name__ == "__main__":
    main()
