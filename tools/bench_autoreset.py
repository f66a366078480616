"""Cost of resetting finished environments: config C2 (two Ants, Language + tag-distance reward + distance done,
maxSteps 1024) at 4096 and 65 536 envs, timed over two full episodes from reset, for
  fused  `autoReset`: the step kernel resets finished envs in the same launch
  pool   `autoReset` with `startStates`: a 1024-row pool of states from a random rollout, drawn per reset in the kernel
  loop   today's policy loop: step(), then reset(mask=term["__all__"] | trunc["__all__"]) every step (no host check)
  step   step() alone, never resetting (the floor)
Two schedules: `sync` (every env starts at step 0, so all of them truncate on the same step, which is also timed on its
own) and `staggered` (resetNoise 0.05, per-env step counters start uniformly in [0, maxSteps), so about N / 1025
envs end an episode on every step).  Every step goes through MuJoCoRL.step with one fixed action tensor.  Timing: CUDA
events on the stepping stream around the whole window, ended by a synchronise, after warm-up steps; the L2 is NOT
flushed (one timed region, as in a real rollout; bench.py's `episode` protocol).  Also times one reset of all envs:
`reset()` against `reset(options={"qpos", "qvel"})` from rows already on the device (mean of 50 calls).  Prints the GPU
name and power limit from the same run, one JSON line per measurement and tables.

usage: python tools/bench_autoreset.py [--envs 4096 65536] [--warmup 20] [--out FILE]
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
from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL  # noqa: E402

LV = os.path.join(ROOT, "tests", "levels")
MAX_STEPS = 1024


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        out = ""
    return name, out or "unknown"


def make_env(n, mode, staggered, pool=None):
    extra = {"startStates": {"qpos": pool[0], "qvel": pool[1]}} if mode == "pool" else {}
    return MuJoCoRL({**extra, "xmlPath": os.path.join(LV, "two_ants.xml"), "infoJson": os.path.join(LV, "info_2A.json"),
                     "agents": ["sender", "receiver"], "environmentDynamics": [P.Language],
                     "rewardFunctions": [P.tag_distance_reward], "doneFunctions": [P.distance_done], "num_envs": n,
                     "maxSteps": MAX_STEPS, "seed": 77, "autoReset": mode in ("fused", "pool"), "resetNoise": 0.05 if staggered else 0.0})


def rollout_states(rows, steps=50):
    """qpos / qvel rows of a C2 rollout with random actions (the start-state pool)"""
    env = make_env(rows, "step", False)
    env.reset()
    for _ in range(steps):
        env.step(env.sample_actions())
    return env.batch.qpos[:, :env.model.nq].clone(), env.batch.qvel[:, :env.model.nv].clone()


def time_resets(n, calls=50):
    env = make_env(n, "step", False)
    qpos, qvel = rollout_states(n, 20)
    out = {"envs": n}
    for name, fn in (("reset", lambda: env.reset()), ("reset_options", lambda: env.reset(options={"qpos": qpos, "qvel": qvel}))):
        for _ in range(5):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(calls):
            fn()
        e1.record()
        torch.cuda.synchronize()
        out[f"ms_{name}"] = round(e0.elapsed_time(e1) / calls, 5)
    return out


def run(n, mode, staggered, warmup, pool=None):
    env = make_env(n, mode, staggered, pool)
    b = env.batch
    act = env.sample_actions()
    A = len(env.agents)

    def one():
        obs, rew, term, trunc, info = env.step(act)
        if mode == "loop":
            env.reset(mask=b.term[:, A].view(torch.bool) | b.trunc[:, A].view(torch.bool))

    env.reset()
    for _ in range(warmup):
        one()
    env.reset()
    if staggered:
        g = torch.Generator(device=env.device).manual_seed(5)
        b.timestep.copy_(torch.randint(0, MAX_STEPS, (n,), generator=g, device=env.device, dtype=torch.int32))
    steps = 2 * (MAX_STEPS + 1)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
    torch.cuda.synchronize()
    ev[0].record()
    for k in range(steps):
        if k == MAX_STEPS - 1:
            ev[2].record()
        if k == MAX_STEPS:   # sync schedule: every env truncates on this step
            ev[3].record()
            ev[4].record()
        one()
        if k == MAX_STEPS:
            ev[5].record()
    ev[1].record()
    torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[1]) / steps
    res = {"envs": n, "mode": mode, "schedule": "staggered" if staggered else "sync", "steps": steps,
           "ms_per_step": round(ms, 5), "agent_steps_per_s": round(n * A / ms * 1e3, 1)}
    if not staggered:
        res["ms_plain_step_before"] = round(ev[2].elapsed_time(ev[3]), 5)
        res["ms_all_truncate_step"] = round(ev[4].elapsed_time(ev[5]), 5)
    del env, b
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, nargs="+", default=[4096, 65536])
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_autoreset: needs a CUDA device")
    name, plimit = device_info()
    print(json.dumps({"device": name, "power_limit": plimit, "l2": "not flushed"}))
    rows = []
    pool = rollout_states(1024)
    for n in args.envs:
        for staggered in (False, True):
            for mode in ("fused", "pool", "loop", "step"):
                r = run(n, mode, staggered, args.warmup, pool)
                print(json.dumps(r), flush=True)
                rows.append(r)
    print(f"\n{name}, power limit {plimit}; ms/step (M agent-steps/s) over {2 * (MAX_STEPS + 1)} steps from reset")
    print("| envs | schedule | (a) fused autoReset | (a') (a) + 1024-row pool | (b) step + reset(mask) | (c) step alone | "
          "all-truncate step (a) / (a') / (b) / (c) |")
    print("|---|---|---|---|---|---|---|")
    for n in args.envs:
        for sched in ("sync", "staggered"):
            r = {x["mode"]: x for x in rows if x["envs"] == n and x["schedule"] == sched}
            cell = lambda m: f"{r[m]['ms_per_step']:.4f} ({r[m]['agent_steps_per_s'] / 1e6:.1f})"
            single = " / ".join(f"{r[m]['ms_all_truncate_step']:.3f}" for m in ("fused", "pool", "loop", "step")) if sched == "sync" else "-"
            print(f"| {n} | {sched} | {cell('fused')} | {cell('pool')} | {cell('loop')} | {cell('step')} | {single} |")
    resets = []
    for n in args.envs:
        r = time_resets(n)
        print(json.dumps(r), flush=True)
        resets.append(r)
    print("\n| envs | reset() ms | reset(options={qpos, qvel}) ms |")
    print("|---|---|---|")
    for r in resets:
        print(f"| {r['envs']} | {r['ms_reset']:.4f} | {r['ms_reset_options']:.4f} |")
    if args.out:
        with open(args.out, "w") as fh:
            json.dump({"device": name, "power_limit": plimit, "rows": rows, "resets": resets}, fh, indent=1)


if __name__ == "__main__":
    main()
