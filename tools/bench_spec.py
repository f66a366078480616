"""Generic vs model-specialised step kernel (DESIGN §7a): the same configs built twice in one process, once with
MJB_SPEC_GENERIC, stepped with the same actions and compared buffer for buffer (bit for bit), then timed alternately with
bench.py's hygiene (settled state, L2 flushed before every step, CUDA events around the kernel).

    python tools/bench_spec.py [--steps 30] [--repeats 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
LEVELS = os.path.join(ROOT, "tests", "levels")

import torch  # noqa: E402

from mujoco_rl_environment_wrapper_b200 import _lib as L  # noqa: E402
from mujoco_rl_environment_wrapper_b200 import mujoco_rl as R  # noqa: E402
from mujoco_rl_environment_wrapper_b200 import plugins as P  # noqa: E402


def make_env(cfg, generic):
    """MuJoCoRL(cfg); with `generic` its batches run the generic step kernel (MJB_SPEC_GENERIC)"""
    if not generic:
        return R.MuJoCoRL(dict(cfg))
    base = R.Batch

    class GenericBatch(base):
        def __init__(self, model, spec, *a, **kw):
            spec = L.EnvSpec.from_buffer_copy(spec)
            spec.flags |= L.SPEC_GENERIC
            super().__init__(model, spec, *a, **kw)

    R.Batch = GenericBatch
    try:
        return R.MuJoCoRL(dict(cfg))
    finally:
        R.Batch = base


def configs():
    two = dict(xmlPath=os.path.join(LEVELS, "two_ants.xml"), infoJson=os.path.join(LEVELS, "info_2A.json"), agents=["sender", "receiver"])
    c2 = dict(two, environmentDynamics=[P.Language], rewardFunctions=[P.tag_distance_reward], doneFunctions=[P.distance_done])
    ant = dict(xmlPath=os.path.join(LEVELS, "ant_rk4.xml"), agents=["torso"], rewardFunctions=[P.ant_reward_function])
    return [
        ("C2", c2, 4096, 300),
        ("C2-65536", c2, 65536, 300),
        ("C1", dict(xmlPath=os.path.join(LEVELS, "one_ant_arena.xml"), agents=["sender"]), 16384, 300),
        ("C3-physics", dict(ant, skipFrames=1), 65536, 200),
        ("C4-3sensors", dict(xmlPath=os.path.join(LEVELS, "two_ants_touch_acc.xml"), agents=["sender", "receiver"], freeJoint=True,
                             skipFrames=5), 16384, 60),
        ("C5", dict(two, environmentDynamics=[P.PickUpDynamic]), 32768, 300),
    ]


def buffers(env):
    b = env.batch
    out = {k: v for k, v in b.buf.items()}
    for k in ("final_obs", "params"):
        t = getattr(b, k, None)
        if isinstance(t, torch.Tensor):
            out[k] = t
    return out


def differing(a, b):
    ba, bb = buffers(a), buffers(b)
    return sorted(k for k in ba if not torch.equal(ba[k].view(torch.uint8) if ba[k].dtype != torch.uint8 else ba[k],
                                                   bb[k].view(torch.uint8) if bb[k].dtype != torch.uint8 else bb[k]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--only", default="")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    res = {"card": card, "l2": "flushed before every step (256 MiB write, outside the events)", "configs": []}
    for name, cfg, n, settle in configs():
        if args.only and name not in args.only.split(","):
            continue
        cfg = dict(cfg, num_envs=n, seed=1234, maxSteps=1024, device=dev)
        envs = {"generic": make_env(cfg, True), "specialised": make_env(cfg, False)}
        geo = envs["specialised"].batch.geometry()
        assert geo["specialised"], geo["spec_reason"]
        assert not envs["generic"].batch.geometry()["specialised"]
        pool = torch.stack([envs["generic"].sample_actions() for _ in range(32)])
        ad = envs["generic"]._act_dim
        for e in envs.values():
            e.reset()
        for k in range(settle):
            for e in envs.values():
                e.batch.actions[:, :, :ad].copy_(pool[k % 32])
                e.batch.step()
        torch.cuda.synchronize(dev)
        diff = differing(envs["generic"], envs["specialised"])
        times = {"generic": [], "specialised": []}
        for r in range(args.repeats):
            for kind in ("generic", "specialised"):
                b = envs[kind].batch
                for k in range(3):
                    b.actions[:, :, :ad].copy_(pool[k]); b.step()
                ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
                torch.cuda.synchronize(dev)
                for k in range(args.steps):
                    flush.zero_()
                    b.actions[:, :, :ad].copy_(pool[k % 32])
                    ev[k][0].record()
                    b.step()
                    ev[k][1].record()
                torch.cuda.synchronize(dev)
                times[kind].append(sum(a.elapsed_time(z) for a, z in ev) / args.steps)
        # both sides took the same steps in the timing loop too
        diff_after = differing(envs["generic"], envs["specialised"])
        gm, sm = min(times["generic"]), min(times["specialised"])
        rec = {"name": name, "num_envs": n, "settle": settle, "kernel_ms": times, "speedup_best": gm / sm,
               "speedup_median": sorted(times["generic"])[len(times["generic"]) // 2] / sorted(times["specialised"])[len(times["specialised"]) // 2],
               "differing_after_settle": diff, "differing_after_timing": diff_after, "spec_compile_ms": geo["spec_compile_ms"],
               "ncon_mean": float(envs["specialised"].batch.ncon.float().mean())}
        print(json.dumps(rec), flush=True)
        res["configs"].append(rec)
        del envs
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps({"card": card}))


if __name__ == "__main__":
    main()
