#!/usr/bin/env python
"""bench.py — agent-steps/s of the batched MuJoCoRL.step hot path on B200 (BASELINE.json metric).

Headline workload (config C2, BASELINE.json configs[1], SURVEY.md 8d): benchmarking/levels/MultiAgentModel.xml,
agents sender + receiver, Language dynamic + tag-distance reward + done, freeJoint = False, skipFrames = 1,
4096 envs PER GPU (weak scaling: envs shard by index, no collective on the step path), synthetic random actions
(pre-generated on the device, one device-to-device copy per step).

One "step" = one `MuJoCoRL.step` for every env of the rank = ONE fused kernel launch.
  value    device-resident throughput, per-step CUDA events on the launching stream, L2 flushed between steps
  e2e      the same through the C-ABI host-buffer call (mjb_step_host): pinned H2D of the actions and D2H of
           obs / rewards / flags inside the timed region
  roofline algorithmic HBM bytes per launch / kernel time vs MEASURED_PEAKS.json (the physics step is latency /
           issue bound, so its fraction is tiny by construction — DESIGN.md; the literal skipFrames = 0 step in
           `configs` IS HBM bound)
  configs  every other BASELINE.json config with the same timing hygiene: C1, C2 at 65536 total envs, C2 over a
           whole 1024-step episode from reset (the reference's protocol, fps_custom_env.py:52-68), C3 literal and
           physics at 65536 TOTAL envs split over the ranks (strong scaling), C4, C5 at 32768 total
  cpu_baseline / --impl reference: the fp64 oracle + reference-order host loop on the host cores
           (kind "port": the reference's MuJoCo dependency is not installable here).
"""
import argparse
import hashlib
import json
import multiprocessing as mp
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
LEVELS = os.path.join(ROOT, "tests", "levels")
ENVS_PER_GPU = int(os.environ.get("MJB_BENCH_ENVS", "4096"))
SETTLE = int(os.environ.get("MJB_BENCH_SETTLE", "300"))
DUMP_LIMIT = 64 << 20   # bytes of --dump-outputs files in all
WORKLOAD = "C2: MultiAgentModel.xml, 2 agents, Language + tag-distance reward + done, ctrl mode, skipFrames=1"
L2_NOTE = "flushed between steps (256 MiB write, outside the per-step events)"


def shared_config():
    """the `config` object of BOTH arms (the driver compares them)"""
    return {"workload": WORKLOAD, "envs_per_gpu": ENVS_PER_GPU, "agents": 2, "l2": L2_NOTE,
            "state": f"settled for {SETTLE} steps before timing"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


def csrc_sha16():
    """fingerprint of the kernel sources: instruction counts taken from an ncu capture are only used while they
    still describe the code that is running"""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "mujoco_rl_environment_wrapper_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cuh", ".cu", ".h", ".cpp")):
            h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def algorithmic_bytes_per_env_step(nq, nv, nu, nsens, n_agents, act_dim, obs_dim, nprobe):
    """SURVEY.md 8d: fp32 state read + written once, actions read, obs / reward / flags written, plugin store
    read + written, qacc warm start read + written."""
    read = 4 * (nq + nv + nu + nv + n_agents * act_dim) + 28
    write = 4 * (nq + nv + nu + nv + nsens + n_agents * obs_dim + n_agents + 4 * nprobe) + 2 * (n_agents + 1) + 4 + 16
    return read + write


def literal_bytes_per_env_step(nq, nv, nu, nsens, n_agents, act_dim, obs_dim, nprobe, free_joint):
    """skipFrames = 0 (no physics): qpos / qvel / ctrl / sensordata / actions / positions / store / counter read once;
    obs, the action-modified array (qvel or ctrl), reward, flags, store and counter written once."""
    store = 4 * n_agents * (8 + 4)
    read = 4 * (nq + nv + nu + nsens + n_agents * act_dim + 4 * nprobe + 1) + store
    write = 4 * (n_agents * obs_dim + (nv if free_joint else nu) + n_agents + 1) + 2 * (n_agents + 1) + store
    return read + write


def dump_outputs(out_dir, arrays, limit=DUMP_LIMIT):
    """Writes `arrays` ({name: array with one row per env}) as out_dir/<name>.npy, float64 kept, everything else as
    float32, plus env_index.npy, the envs the rows belong to.  When all envs would take more than `limit` bytes, a
    fixed seeded sample of envs is written, the same for every build, so that two builds compare row for row."""
    import numpy as np
    arrays = {k: np.asarray(v, dtype=np.float64 if np.asarray(v).dtype == np.float64 else np.float32) for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    per_env = 8 + sum(a.nbytes for a in arrays.values()) // n
    keep = (limit - 4096 * (len(arrays) + 1)) // per_env   # leaves room for each file's .npy header (128 bytes)
    rows = np.arange(n) if n <= keep else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "env_index.npy"), rows.astype(np.float64))
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a[rows])


# ------------------------------------------------------------------------------------------------
# CPU arm: oracle physics + reference-order host loop, one env per process
_CPU_ENV = None


def _cpu_env(seed):
    global _CPU_ENV
    if _CPU_ENV is None:
        sys.path.insert(0, ROOT)
        import numpy as np
        from mujoco_rl_environment_wrapper_b200 import _lib as L
        from mujoco_rl_environment_wrapper_b200.tables import Tables
        from oracle import host_loop as H
        text = open(os.path.join(LEVELS, "two_ants.xml")).read()
        model = L.Model(text)
        agents = ["sender", "receiver"]
        tables = Tables(text, model, agents, False)

        def resolve(name):
            b = model.name2id(L.OBJ_BODY, name)
            return (1, b) if b >= 0 else (5, model.name2id(L.OBJ_GEOM, name))
        rng = np.random.default_rng(seed)
        env = H.OracleEnv(model, tables, agents, dynamics=[H.Language], reward_functions=[H.tag_distance_reward],
                          done_functions=[H.distance_done], targets=["choice_1", "choice_2"],
                          draw=lambda a, k: int(rng.integers(0, 1 << 30)), resolve=resolve)
        env.reset({a: np.zeros(9) for a in agents})
        _CPU_ENV = (env, rng, agents, np)
    return _CPU_ENV


def _cpu_worker(args):
    seed, seconds = args
    env, rng, agents, np = _cpu_env(seed)
    steps, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        act = {a: np.concatenate([rng.uniform(-1, 1, 8), rng.uniform(0, 3, 1)]) for a in agents}
        env.step(act)
        steps += 1
        if env.timestep >= 1024:
            env.reset({a: np.zeros(9) for a in agents})
    return steps, time.perf_counter() - t0


def cpu_arm(seconds, pool, cores):
    res = pool.map(_cpu_worker, [(1000 + i, seconds) for i in range(cores)], chunksize=1)
    env_steps = sum(r[0] for r in res)
    wall = max(r[1] for r in res)
    return 2.0 * env_steps / wall, env_steps


def make_pool():
    cores = os.cpu_count() or 1
    pool = mp.get_context("spawn").Pool(cores)
    pool.map(_cpu_worker, [(1000 + i, 0.05) for i in range(cores)], chunksize=1)  # build the envs
    return pool, cores


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import build_oracle
    build_oracle()
    pool, cores = make_pool()
    per_step_s = min(10.0, max(0.05, 100.0 / max(1, args.steps + args.warmup)))
    vals = []
    for i in range(args.warmup + args.steps):
        v, n = cpu_arm(per_step_s, pool, cores)
        if i >= args.warmup:
            vals.append(v)
    pool.close()
    value = sum(vals) / len(vals)
    sample = f"{cores} processes x 1 env, {per_step_s:.2f} s of random-action steps per timed step, {WORKLOAD}"
    print(json.dumps({
        "impl": "reference", "metric": "agent-steps/sec", "value": value, "unit": "agent-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_step_s * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": shared_config(),
        "detail": {"envs_per_process": 1, "processes": cores, "note": "config.l2 / config.state describe the GPU arm; the CPU arm runs "
                   "one env per host process from reset, 1024-step episodes"},
        "cpu_baseline": {"value": value, "unit": "agent-steps/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "agent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "restated-CPU (fp64 oracle + reference-order Python host loop), NOT MuJoCo: mujoco==2.3.3 is not installable here",
    }))


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU every 10 ms on a thread (NVML), DURING the timed region."""
    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, index):
        self.index, self.sm, self.reasons, self.max_sm, self._stop, self._thr = index, [], set(), None, False, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nv = None
            return
        self._thr = threading.Thread(target=self._run, daemon=True)
        self._thr.start()

    def _run(self):
        nv = self._nv
        while not self._stop:
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for name, bit in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.01)

    def stop(self):
        self._stop = True
        if self._thr:
            self._thr.join(timeout=1.0)
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_sm, "reasons": sorted(self.reasons),
                "samples": len(sm)}


def level(name):
    return os.path.join(LEVELS, name)


def config_table(P):
    """(name, workload text, MuJoCoRL config, env count, 'total' | 'per_gpu', settle steps, protocol)"""
    two = dict(xmlPath=level("two_ants.xml"), infoJson=level("info_2A.json"), agents=["sender", "receiver"])
    c2 = dict(two, environmentDynamics=[P.Language], rewardFunctions=[P.tag_distance_reward], doneFunctions=[P.distance_done])
    ant = dict(xmlPath=level("ant_rk4.xml"), agents=["torso"], rewardFunctions=[P.ant_reward_function])
    return [
        ("C1", "SingleAgentModel.xml, 1 agent, ctrl mode, skipFrames=1, no plugins", dict(xmlPath=level("one_ant_arena.xml"), agents=["sender"]),
         16384, "per_gpu", 300, "settled"),
        ("C2-65536", WORKLOAD, c2, 65536, "total", 300, "settled"),
        ("C2-episode", WORKLOAD + "; reset + 1024 steps timed as one region (fps_custom_env.py:52-68)", c2, ENVS_PER_GPU, "per_gpu", 0, "episode"),
        ("C3-literal", "Ant.xml, freeJoint, skipFrames=0 (no physics), ant reward: fps_custom_env.py:39-48 verbatim", dict(ant, freeJoint=True, skipFrames=0),
         65536, "total", 10, "settled"),
        ("C3-physics", "Ant.xml, ctrl mode, RK4, skipFrames=1, ant reward", dict(ant, skipFrames=1), 65536, "total", 200, "settled"),
        ("C4-rangefinder", "sensor_levels/Model3.xml (free box + rangefinder), freeJoint, skipFrames=5", dict(xmlPath=level("box_rangefinder.xml"), agents=["receiver"],
                                                                                                     freeJoint=True, skipFrames=5), 16384, "per_gpu", 60, "settled"),
        ("C4-3sensors", "MultiAgentModel3Sensors.xml (rangefinder + touch + accelerometer), freeJoint, skipFrames=5",
         dict(xmlPath=level("two_ants_touch_acc.xml"), agents=["sender", "receiver"], freeJoint=True, skipFrames=5), 16384, "per_gpu", 60, "settled"),
        ("C5", "MultiAgentModel.xml, 2 agents, Pick_Up dynamic, ctrl mode, skipFrames=1", dict(two, environmentDynamics=[P.PickUpDynamic]), 32768, "total", 300, "settled"),
    ]


def run_ours(args):
    import numpy as np
    import torch
    from mujoco_rl_environment_wrapper_b200 import dist as D
    from mujoco_rl_environment_wrapper_b200 import plugins as P
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL
    rank, local, world = D.init_from_env()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    peak, which = peaks()
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    sha = csrc_sha16()
    counts = {}
    cp = os.path.join(ROOT, "profiles", "r02_counts.json")
    if os.path.exists(cp):
        cj = json.load(open(cp))
        if cj.get("csrc_sha16") == sha:   # a stale capture says nothing about the kernel that is running now
            counts = cj.get("configs", {})

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize(dev)

    def action_pool(env, n=16):
        return torch.stack([env.sample_actions() for _ in range(n)])

    def timed_steps(env, pool, steps, warmup):
        """`steps` timed steps: L2 flushed before each, one event pair per step (action copy + kernel) and one around
        the kernel alone; returns (ms per step, kernel ms per step), each the max over ranks"""
        b, ad = env.batch, env._act_dim
        for k in range(warmup):
            b.actions[:, :, :ad].copy_(pool[k % len(pool)]); b.step()
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(steps)]
        barrier()
        for k in range(steps):
            flush.zero_()                                      # L2 flush, outside the per-step events
            ev[k][0].record()
            b.actions[:, :, :ad].copy_(pool[k % len(pool)])    # this step's synthetic actions (device to device)
            ev[k][1].record()
            b.step()                                           # the fused kernel
            ev[k][2].record()
            ev[k][3].record()
        barrier()
        step_ms = sum(e[0].elapsed_time(e[3]) for e in ev) / steps
        kern_ms = sum(e[1].elapsed_time(e[2]) for e in ev) / steps
        return D.max_over_ranks(step_ms, dev), D.max_over_ranks(kern_ms, dev)

    def issue_record(name, kern_ms, n_envs, mhz):
        c = counts.get(name)
        if not c or not c.get("warp_instructions_per_env"):
            return None
        inst = c["warp_instructions_per_env"] * n_envs
        peak_ips = sms * 4 * mhz * 1e6
        return {"warp_instructions_per_launch": inst, "achieved_ginst_s": inst / (kern_ms * 1e-3) / 1e9, "peak_ginst_s": peak_ips / 1e9,
                "frac": inst / (kern_ms * 1e-3) / peak_ips,
                "note": f"executed warp instructions per env from the ncu capture of THESE sources (csrc sha {sha}, {c.get('envs')} envs), "
                        "time and clock live; 4 issue slots per SM per cycle"}

    # ================================ headline: C2, weak scaling =========================================================
    N = ENVS_PER_GPU
    env = MuJoCoRL({"xmlPath": level("two_ants.xml"), "infoJson": level("info_2A.json"),
                    "agents": ["sender", "receiver"], "skipFrames": 1, "maxSteps": 1024, "num_envs": N,
                    "seed": 1234 + 1000 * rank, "device": dev, "environmentDynamics": [P.Language],
                    "rewardFunctions": [P.tag_distance_reward], "doneFunctions": [P.distance_done]})
    b = env.batch
    A, act_dim = 2, env._act_dim
    pool = action_pool(env, 32)
    env.reset()
    # settle onto the floor so that the timed steps carry contacts (whole episodes are timed in configs["C2-episode"])
    for k in range(SETTLE):
        b.actions[:, :, :act_dim].copy_(pool[k % 32])
        b.step()
    torch.cuda.synchronize(dev)
    clocks = ClockSampler(local)
    clocks.start()
    launches0 = b.launch_count
    t_wall0 = time.perf_counter()
    warm = max(3, args.warmup)
    step_ms, kern_ms = timed_steps(env, pool, args.steps, warm)
    t_wall = time.perf_counter() - t_wall0
    launches = b.launch_count - launches0 - warm
    if args.dump_outputs:   # what the last timed step returned (the end-to-end arm below steps on)
        obs_dim = max(env._spec.obs_dim[a] for a in range(A))
        last = {"obs": b.obs[:, :, :obs_dim].cpu(), "reward": b.reward.cpu(), "term": b.term.cpu(), "trunc": b.trunc.cpu()}

    # ---- end-to-end arm: C-ABI host-buffer call, pinned H2D / D2H inside the timed region
    h_act, h_obs, h_rew, h_term, h_trunc = b.host_arrays()
    # each step's actions arrive in page-locked host memory (four different buffers in rotation, as a policy's output
    # ring would be); results land in page-locked host arrays
    pinned_keep = [torch.zeros(h_act.shape, dtype=torch.float32, pin_memory=True) for _ in range(4)]
    host_acts = [t.numpy() for t in pinned_keep]
    for k in range(4):
        host_acts[k][:, :, :act_dim] = pool[k].cpu().numpy()
    for k in range(4):
        b.step_host(host_acts[k % 4], h_obs, h_rew, h_term, h_trunc)
    barrier()
    t0 = time.perf_counter()
    for k in range(args.steps):
        b.step_host(host_acts[k % 4], h_obs, h_rew, h_term, h_trunc)
    torch.cuda.synchronize(dev)
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    e2e_ms = D.max_over_ranks(e2e_ms, dev)
    clk = clocks.stop()
    mhz = (clk or {}).get("sm_mhz") or (clk or {}).get("sm_max_mhz") or 1965

    # optional end-of-rollout collective (outside every timed region)
    stats = torch.tensor([float(b.reward.sum()), float(b.term[:, A].sum()), float(b.ncon.float().mean())], device=dev)
    allstats = D.allgather_episode_stats(stats)
    m = env.model
    bytes_env = algorithmic_bytes_per_env_step(m.nq, m.nv, m.nu, m.nsensordata, A, act_dim, 60, b.layout.probe_count)
    head_stats = {"ncon_mean": float(b.ncon.float().mean()), "niter_mean": float(b.niter.float().mean()), "ncon_dropped": int(b.ncon_dropped.sum())}
    geometry = b.geometry()
    del env, b
    torch.cuda.empty_cache()

    # ================================ every other BASELINE config ========================================================
    cfg_steps = max(5, min(args.steps, 30))
    configs = []
    if not args.no_configs:
        for name, text, cfg, count, split, settle, protocol in config_table(P):
            n_gpu = count if split == "per_gpu" else max(1, count // world)
            total = n_gpu * world
            e = MuJoCoRL(dict(cfg, num_envs=n_gpu, seed=4321 + 1000 * rank, device=dev, maxSteps=1024))
            bb, nA, ad = e.batch, len(e.agents), e._act_dim
            pl = action_pool(e, 16)
            mm = e.model
            obs_dim = max(e._spec.obs_dim[a] for a in range(nA))
            if protocol == "episode":
                e.reset()
                for k in range(3):
                    bb.actions[:, :, :ad].copy_(pl[k]); bb.step()
                barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ncon_acc = torch.zeros((), device=dev)
                e0.record()
                e.reset()
                for k in range(1024):
                    bb.actions[:, :, :ad].copy_(pl[k % 16]); bb.step()
                    if k % 128 == 127:
                        ncon_acc += bb.ncon.float().mean()
                e1.record()
                barrier()
                ms = D.max_over_ranks(e0.elapsed_time(e1) / 1024, dev)
                kms, ncon_mean = None, float(ncon_acc) / 8
                l2 = "not flushed (one timed region of reset + 1024 steps; 4096 envs' rows stay L2 resident, as in a real rollout)"
            else:
                e.reset()
                for k in range(settle):
                    bb.actions[:, :, :ad].copy_(pl[k % 16]); bb.step()
                ms, kms = timed_steps(e, pl, cfg_steps, 3)
                ncon_mean, l2 = float(bb.ncon.float().mean()), L2_NOTE
            literal = int(cfg.get("skipFrames", 1)) == 0
            if literal:
                by = literal_bytes_per_env_step(mm.nq, mm.nv, mm.nu, mm.nsensordata, nA, ad, obs_dim, bb.layout.probe_count, bool(cfg.get("freeJoint")))
            else:
                by = algorithmic_bytes_per_env_step(mm.nq, mm.nv, mm.nu, mm.nsensordata, nA, ad, obs_dim, bb.layout.probe_count)
            st = torch.tensor([ncon_mean, float(bb.niter.float().mean()), float(bb.ncon_dropped.sum())], device=dev)
            st = D.allgather_episode_stats(st).mean(dim=0).cpu().tolist() if world > 1 else st.cpu().tolist()
            gb = by * n_gpu / ((kms or ms) * 1e-3) / 1e9
            configs.append({
                "name": name, "workload": text, "scaling": "strong" if split == "total" else "weak", "envs_total": total, "envs_per_gpu": n_gpu,
                "agents": nA, "skip_frames": int(cfg.get("skipFrames", 1)), "protocol": protocol, "l2": l2, "steps": 1024 if protocol == "episode" else cfg_steps,
                "ms_per_step": ms, "kernel_ms": kms, "agent_steps_per_s": total * nA / (ms * 1e-3),
                "ncon_mean": st[0], "niter_mean": None if literal else st[1], "ncon_dropped": int(st[2] * (world if world > 1 else 1)),
                "hbm": {"algorithmic_bytes_per_env_step": by, "achieved_GBps": gb, "frac": gb / peak, "bound": "hbm" if literal else "issue/latency"},
                "issue": issue_record(name, kms or ms, n_gpu, mhz), "geometry": bb.geometry()})
            del e, bb
            torch.cuda.empty_cache()

    if rank == 0:
        traffic = None
        c2 = counts.get("C2")
        if c2 and c2.get("envs") == N:
            traffic = c2.get("dram_bytes")
        achieved = bytes_env * N / (kern_ms * 1e-3) / 1e9
        agent_steps = N * A * world
        out = {
            "metric": "agent-steps/sec", "value": agent_steps / (step_ms * 1e-3), "unit": "agent-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": step_ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": shared_config(),
            "detail": dict(head_stats, geometry=geometry, wall_ms_per_step_incl_flush=t_wall * 1e3 / (args.steps + warm), csrc_sha16=sha),
            "e2e": {"value": agent_steps / (e2e_ms * 1e-3), "unit": "agent-steps/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": int(h_act.nbytes), "d2h_bytes_per_step": int(h_obs.nbytes + h_rew.nbytes + h_term.nbytes + h_trunc.nbytes)},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "peak_source": which, "algorithmic_bytes_per_env_step": bytes_env, "kernel_ms": kern_ms,
                         "note": "physics-on step is issue/latency bound (SURVEY 8d): see profiles/ for issue-slot and stall evidence; the HBM-bound "
                                 "step is configs[C3-literal]",
                         "issue": issue_record("C2", kern_ms, N, mhz)},
            "clocks": clk,
            "episode_stats_allgather": allstats.cpu().tolist(),
            "configs": configs,
        }
        if world == 1 and not args.no_cpu:
            from oracle import build_oracle
            build_oracle()
            cpool, cores = make_pool()
            v, n = cpu_arm(12.0, cpool, cores)
            cpool.close()
            out["cpu_baseline"] = {"value": v, "unit": "agent-steps/s", "cores": cores, "kind": "port",
                                   "sample": f"{cores} processes x 1 env x 12 s of the same workload ({n} env-steps), fp64 oracle + reference-order host loop"}
        print(json.dumps(out))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {k: v.numpy() for k, v in last.items()})
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-configs", action="store_true", help="headline config only")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write obs / reward / term / trunc of the last timed headline step as "
                    "DIR/<name>.npy (rank 0's envs), to compare two builds on the same inputs")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
