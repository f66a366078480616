"""Cost of the frame, velocity and joint sensors (DESIGN §5f), step time for
  C2      two Ants (two_ants.xml), Language + tag-distance reward + distance done, skipFrames 1
  C2+IMU  the same scene with a torso IMU per ant (two_ants_imu.xml: gyro, velocimeter, accelerometer, framequat, four joint
          sensors and a foot velocity per ant), observed by its agent ("sensors"), and the same without the two
          accelerometers ("noacc": only the new pass, no acceleration-stage sensor)
at 4096 and 65 536 envs, and
  box     box_imu.xml without its sensors, freeJoint actions, skipFrames 5, four envs per warp
  box+27  box_imu.xml with its 27 sensors (86 floats)
at 16 384 envs.  The sensor-free variants are the same XML with the <sensor> block removed, so the two members of a pair differ
only in their sensors.  Every step goes through MuJoCoRL.step with one fixed action tensor.  Timing: CUDA events on the
stepping stream around `--steps` steps after `--warmup` steps, ended by a synchronise; the L2 is not flushed.  The members
of a pair alternate within each repeat.  Also prints the launch geometry (grid, env-warps per CTA, shared memory per CTA),
and the GPU name and power limit from the same run; one JSON line per measurement.

usage: python tools/bench_sensors.py [--steps 300] [--warmup 30] [--repeats 3] [--out FILE]
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from mujoco_rl_environment_wrapper_b200 import plugins as P  # noqa: E402
from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL  # noqa: E402

LV = os.path.join(ROOT, "tests", "levels")
SLV = os.path.join(ROOT, "tests", "sensor_levels")
# (label, envs, with sensors (tests/sensor_levels), without (tests/levels))
CASES = [("C2", 4096, "two_ants_imu.xml", "two_ants.xml"), ("C2", 65536, "two_ants_imu.xml", "two_ants.xml"),
         ("box_imu", 16384, "box_imu.xml", None)]


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        out = ""
    return name, out or "unknown"


def without_sensors(xml_name, tmp):
    text = re.sub(r"<sensor>.*?</sensor>", "", open(os.path.join(SLV, xml_name)).read(), flags=re.S)
    path = os.path.join(tmp, "nosensors_" + xml_name)
    open(path, "w").write(text)
    return path


def without_accelerometers(xml_name, tmp):
    text = re.sub(r"\s*<accelerometer [^>]*/>", "", open(os.path.join(SLV, xml_name)).read())
    path = os.path.join(tmp, "noacc_" + xml_name)
    open(path, "w").write(text)
    return path


def make_env(path, n):
    if "box" in os.path.basename(path):
        cfg = {"xmlPath": path, "agents": ["receiver"], "freeJoint": True, "skipFrames": 5}
    else:
        cfg = {"xmlPath": path, "infoJson": os.path.join(LV, "info_2A.json"), "agents": ["sender", "receiver"],
               "environmentDynamics": [P.Language], "rewardFunctions": [P.tag_distance_reward], "doneFunctions": [P.distance_done]}
    env = MuJoCoRL({**cfg, "num_envs": n, "seed": 77})
    env.reset()
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
    assert torch.isfinite(env.batch.qpos).all() and torch.isfinite(env.batch.sensordata).all()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=30)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sensors: needs a CUDA device")
    gpu, power = device_info()
    rows = []
    with tempfile.TemporaryDirectory() as tmp:
        for label, n, with_s, without in CASES:
            paths = {"sensors": os.path.join(SLV, with_s),
                     "none": os.path.join(LV, without) if without else without_sensors(with_s, tmp)}
            if "two_ants" in with_s:   # the IMU without its accelerometers: what the new pass alone costs
                paths["noacc"] = without_accelerometers(with_s, tmp)
            envs = {k: make_env(p, n) for k, p in paths.items()}
            times = {k: [] for k in envs}
            for _ in range(args.repeats):
                for k in envs:
                    times[k].append(time_steps(envs[k], args.steps, args.warmup))
            for k in envs:
                geo = envs[k].batch.geometry()
                r = {"gpu": gpu, "power_limit": power, "case": label, "envs": n, "variant": k,
                     "nsensordata": envs[k].model.nsensordata, "ms_per_step": [round(t, 5) for t in times[k]],
                     "ms_per_step_min": round(min(times[k]), 5), "warps_per_cta": geo["warps_per_cta"], "grid": geo["grid"],
                     "smem_bytes": geo["smem_bytes"]}
                rows.append(r)
                print(json.dumps(r), flush=True)
            del envs
            torch.cuda.empty_cache()
    print(f"\n{gpu}, power limit {power}; ms per step (min over {args.repeats} alternating repeats of {args.steps} steps)")
    print(f"{'case':>8} {'envs':>6} {'variant':>8} {'nsensdata':>9} {'ms/step':>9} {'ratio':>6} {'warps/CTA':>9} {'grid':>6} {'smem/CTA':>9}")
    for r in rows:
        base = next(x for x in rows if x["case"] == r["case"] and x["envs"] == r["envs"] and x["variant"] == "none")["ms_per_step_min"]
        print(f"{r['case']:>8} {r['envs']:>6} {r['variant']:>8} {r['nsensordata']:>9} {r['ms_per_step_min']:>9.4f} {r['ms_per_step_min'] / base:>6.3f} "
              f"{r['warps_per_cta']:>9} {r['grid']:>6} {r['smem_bytes']:>9}")
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rows, f, indent=1)


if __name__ == "__main__":
    main()
