"""Auto-reset (config "autoReset", MJB_SPEC_AUTORESET): a step resets every env whose episode it ended in the same
launch.  Every auto-reset step is compared bit for bit, in every buffer, with the path it replaces: a plain step, then
the finished envs' actions set from a numpy restatement of the documented draw (include/mjb.h, mjb_reset_action), a
masked reset, and the step's reward / term / trunc put back.  The kernel source runs on the host SIMT emulator in both
lane orders, and through libmjb.so on the GPU."""
import ctypes
import os

import numpy as np
import pytest

import emu_harness as E
from common import LEVELS, load_scene, make_spec
from mujoco_rl_environment_wrapper_b200 import _lib as L

U64 = np.uint64


def draw_u32_np(seed, env, agent, counter):
    """csrc/env_kernel.cuh::draw_u32 over numpy arrays (uint64 arithmetic wraps like the kernel's)"""
    env, agent, counter = (np.asarray(x, dtype=U64) for x in (env, agent, counter))
    with np.errstate(over="ignore"):
        z = U64(seed) + U64(0x9E3779B97F4A7C15) * (U64(1) + env) + U64(0xBF58476D1CE4E5B9) * agent + U64(0x94D049BB133111EB) * counter
        z = (z ^ (z >> U64(30))) * U64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> U64(27))) * U64(0x94D049BB133111EB)
        z = z ^ (z >> U64(31))
    return (z >> U64(32)).astype(np.uint32)


def reset_key_np(timestep, qpos0, qvel0):
    """timestep ^ bits(qpos[0]) ^ (bits(qvel[0]) << 13) of the rows the finishing step left"""
    q = np.asarray(qpos0, np.float32).view(np.uint32).astype(U64)
    v = np.asarray(qvel0, np.float32).view(np.uint32).astype(U64)
    t = np.asarray(timestep, np.int32).view(np.uint32).astype(U64)
    return ((t ^ q ^ (v << U64(13))) & U64(0xFFFFFFFF)).astype(np.uint32)


def reset_action_np(seed, env, agent, dim, ep, low, high):
    """the documented draw, in float32 numpy (no fused multiply-add)"""
    u = (draw_u32_np(seed ^ 0x5EEDC0DE, env, 0xC000 + agent * 64 + dim, ep) >> np.uint32(8)).astype(np.float32) * np.float32(2.0 ** -24)
    return np.float32(low) + u * (np.float32(high) - np.float32(low))


def test_reset_action_export_matches_numpy_restatement():
    lib = L.load()
    rng = np.random.default_rng(3)
    for _ in range(200):
        seed, env, agent, dim, ep = int(rng.integers(0, 2 ** 63)), int(rng.integers(0, 1 << 20)), int(rng.integers(0, 8)), \
            int(rng.integers(0, 64)), int(rng.integers(0, 2 ** 32))
        low, high = np.float32(rng.uniform(-5, 1)), np.float32(rng.uniform(1, 7))
        want = reset_action_np(seed, env, agent, dim, ep, low, high)
        got = np.float32(lib.mjb_reset_action(seed, env, agent, dim, ep, low, high))
        assert got.view(np.uint32) == np.asarray(want, np.float32).view(np.uint32)
        assert low <= got < high or got == low


# ---- scenes ------------------------------------------------------------------------------------------------------------
# 2A: Language + tag-distance reward + distance done (threshold between the receiver's two target distances, so that
# about half the episodes end by termination); C1 / 1A: two Ants per warp; S1: four boxes per warp; 3S: freeJoint, skipFrames 5
def scene_spec(scene, max_steps, noise, autoreset, seed=5, skip_frames=1):
    model, tables, agents, fj = load_scene(scene)
    kw = {}
    language = len(agents) > 1 or scene == "C1"
    if language:
        kw["dynamics"] = [(L.DYN_LANGUAGE, 1, 1, 0.0)]
    if scene == "2A":
        kw["targets"] = [(L.OBJ_BODY, model.name2id(L.OBJ_BODY, t)) for t in ("choice_1", "choice_2")]
        kw["rewards"] = [(L.REW_TAG_DISTANCE, 10.0)]
        kw["dones"] = [(L.DONE_DISTANCE_LE, 4.4)]
    spec, keep = make_spec(model, tables, agents, fj, skip_frames=skip_frames, max_steps=max_steps, seed=seed, **kw)
    spec.reset_noise = noise
    low = np.array(list(tables.act_space[agents[0]]["low"]) + ([0.0] if language else []), np.float32)
    high = np.array(list(tables.act_space[agents[0]]["high"]) + ([3.0] if language else []), np.float32)
    if autoreset:
        spec.flags |= L.SPEC_AUTORESET
        for d in range(len(low)):
            spec.act_low[d], spec.act_high[d] = float(low[d]), float(high[d])
    return model, spec, keep, low, high, len(agents)


class EmuSide:
    def __init__(self, model, spec, keep, n, skip_frames, reverse):
        self.eb = E.EmuBatch(model.blob, spec, n, keep)
        self.skip, self.reverse = skip_frames, reverse
        self.final_obs = np.full_like(self.eb.obs, np.nan)
        spec.final_obs = self.final_obs.ctypes.data

    names = property(lambda self: list(self.eb.buf))

    def step(self):
        self.eb.run(E.MODE_STEP, self.skip, reverse=self.reverse)

    def reset(self, mask=None):
        self.eb.run(E.MODE_RESET, mask=mask, reverse=self.reverse)

    def get(self, k):
        return self.final_obs.copy() if k == "final_obs" else self.eb.buf[k].copy()

    def put(self, k, v):
        self.eb.buf[k][...] = v


class GpuSide:
    def __init__(self, model, spec, keep, n, skip_frames, reverse=False):
        from mujoco_rl_environment_wrapper_b200.batch import Batch
        self.b = Batch(model, spec, n, keepalive=keep)
        if spec.flags & L.SPEC_AUTORESET:
            self.b.final_obs.fill_(float("nan"))

    names = property(lambda self: list(self.b.buf))

    def step(self):
        self.b.step()

    def reset(self, mask=None):
        import torch
        self.b.reset(None if mask is None else torch.from_numpy(mask))

    def get(self, k):
        return (self.b.final_obs if k == "final_obs" else self.b.buf[k]).cpu().numpy().copy()

    def put(self, k, v):
        import torch
        self.b.buf[k].copy_(torch.from_numpy(np.ascontiguousarray(v)))


def reference_step(ref, seed, low, high, A):
    """a plain step; then the finished envs get the documented random action and a masked reset; then the step's
    reward / term / trunc are put back.  Returns (finished mask, the step's obs)."""
    ref.step()
    saved = {k: ref.get(k) for k in ("reward", "term", "trunc", "obs")}
    fin = (saved["term"][:, A] | saved["trunc"][:, A]).astype(bool)
    if fin.any():
        acts = ref.get("actions")
        env = np.nonzero(fin)[0]
        ep = reset_key_np(ref.get("timestep")[env], ref.get("qpos")[env, 0], ref.get("qvel")[env, 0])
        drawn = acts.copy()
        for a in range(A):
            for d in range(len(low)):
                drawn[env, a, d] = reset_action_np(seed, env, a, d, ep, low[d], high[d])
        ref.put("actions", drawn)
        ref.reset(fin.astype(np.uint8))
        ref.put("actions", acts)
        for k in ("reward", "term", "trunc"):
            ref.put(k, saved[k])
    return fin, saved["obs"]


def run_against_reference(side, scene, n, steps, noise, max_steps, skip_frames=1, reverse=False, seed=5, plain=False):
    """auto-reset batch vs the reference path, `steps` steps from staggered per-env step counters; returns the number of
    episodes that ended and which envs ended one.  With `plain`, also checks that envs which never finished (with their
    warp neighbours) equal a batch without the flag"""
    model, spec_a, keep_a, low, high, A = scene_spec(scene, max_steps, noise, True, seed, skip_frames)
    _, spec_r, keep_r, _, _, _ = scene_spec(scene, max_steps, noise, False, seed, skip_frames)
    auto = side(model, spec_a, keep_a, n, skip_frames, reverse)
    ref = side(model, spec_r, keep_r, n, skip_frames, reverse)
    sides = [auto, ref]
    if plain:
        _, spec_p, keep_p, _, _, _ = scene_spec(scene, max_steps, noise, False, seed, skip_frames)
        sides.append(side(model, spec_p, keep_p, n, skip_frames, reverse))
    rng = np.random.default_rng(seed)
    e = np.arange(n)
    ts0 = ((e // 4 * 7 + e % 4) % max_steps).astype(np.int32)   # resets hit some copies of a packed warp and not others
    for s in sides:
        s.reset()
        s.put("timestep", ts0)
    names = ref.names
    ended_total, ever = 0, np.zeros(n, bool)
    for t in range(steps):
        act = auto.get("actions")
        act[:, :, :len(low)] = rng.uniform(low, high, (n, A, len(low))).astype(np.float32)
        for s in sides:
            s.put("actions", act)
        before = auto.get("final_obs")
        auto.step()
        if plain:
            sides[2].step()
        fin, obs = reference_step(ref, seed, low, high, A)
        for k in names:
            assert auto.get(k).tobytes() == ref.get(k).tobytes(), (scene, t, k)
        fo = auto.get("final_obs")
        assert fo[fin].tobytes() == obs[fin].tobytes(), (scene, t)
        assert fo[~fin].tobytes() == before[~fin].tobytes(), (scene, t)
        ended_total += int(fin.sum())
        ever |= fin
    if plain:
        # a packed warp (up to four envs) shares the solver's iteration count, so only envs whose whole aligned group of
        # four never finished are independent of the resets around them
        keep = np.repeat(~ever.reshape(-1, 4).any(axis=1), 4)
        for k in names:
            assert auto.get(k)[keep].tobytes() == sides[2].get(k)[keep].tobytes(), (scene, k)
    return ended_total, ever


@pytest.mark.parametrize("reverse", [False, True])
@pytest.mark.parametrize("noise", [0.0, 0.05])
@pytest.mark.parametrize("scene,n,steps,max_steps", [("2A", 8, 7, 5), ("S1", 8, 7, 4), ("C1", 6, 6, 4)])
def test_emulator_autoreset_equals_step_then_masked_reset(scene, n, steps, max_steps, noise, reverse):
    ended, ever = run_against_reference(EmuSide, scene, n, steps, noise, max_steps, reverse=reverse)
    assert ended >= n and ever.all()


def test_emulator_autoreset_ends_episodes_by_termination():
    """2A's distance done ends some episodes before maxSteps: those auto-reset with term set and trunc clear"""
    model, spec, keep, low, high, A = scene_spec("2A", 50, 0.0, True)
    side = EmuSide(model, spec, keep, 8, 1, False)
    side.reset()
    side.step()
    term, trunc = side.get("term"), side.get("trunc")
    hit = term[:, A].astype(bool)
    assert hit.any() and not hit.all() and not trunc[:, A].any()
    assert (side.get("timestep")[hit] == 0).all() and (side.get("timestep")[~hit] == 1).all()


def test_batch_create_refusals_without_gpu():
    """refused before any device work: skipFrames = 0, a missing final_obs buffer"""
    model, spec, keep, low, high, A = scene_spec("2A", 10, 0.0, True)
    lib = L.load()
    h = ctypes.c_void_p()
    spec.skip_frames = 0
    spec.final_obs = 16
    assert lib.mjb_batch_create(model._h, ctypes.byref(spec), 4, 0, None, ctypes.byref(L.Buffers()), ctypes.byref(h)) == -2
    assert b"skip_frames" in lib.mjb_last_error()
    spec.skip_frames, spec.final_obs = 1, None
    assert lib.mjb_batch_create(model._h, ctypes.byref(spec), 4, 0, None, ctypes.byref(L.Buffers()), ctypes.byref(h)) == -2
    assert b"final_obs" in lib.mjb_last_error()


# ---- GPU ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("scene,max_steps,skip_frames", [("2A", 30, 1), ("C1", 28, 1), ("1A", 26, 2), ("3S", 30, 5)])
def test_gpu_autoreset_equals_step_then_masked_reset(scene, max_steps, skip_frames):
    # 20 steps from counters staggered over [0, maxSteps): without 2A's distance done about a third of the envs never finish
    n = 4096
    ended, ever = run_against_reference(GpuSide, scene, n, 20, 0.05 if scene in ("C1", "3S") else 0.0, max_steps,
                                        skip_frames=skip_frames, plain=True)
    assert ended >= n // 2 and (scene == "2A" or (~ever).sum() > n // 8)


def _env(n, **kw):
    from mujoco_rl_environment_wrapper_b200 import plugins as P
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL
    cfg = {"xmlPath": os.path.join(LEVELS, "two_ants.xml"), "infoJson": os.path.join(LEVELS, "info_2A.json"),
           "agents": ["sender", "receiver"], "environmentDynamics": [P.Language], "rewardFunctions": [P.tag_distance_reward],
           "doneFunctions": [P.distance_done], "num_envs": n, "maxSteps": 5, "seed": 11}
    cfg.update(kw)
    return MuJoCoRL(cfg)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 64])
def test_gpu_dropin_infos(n):
    """infos[agent] carries final_observation / _final_observation; the finishing step's values equal those of the
    same env without the flag, and the returned observation is the new episode's first one"""
    import torch
    env, twin = _env(n, autoReset=True), _env(n)
    env.reset()
    twin.reset()
    g = torch.Generator(device=env.device).manual_seed(1)
    ever = torch.zeros(n, dtype=torch.bool, device=env.device)   # envs reset earlier no longer follow the twin
    for t in range(6):
        act = torch.rand((n, 2, 9), generator=g, device=env.device) * torch.tensor([2.0] * 8 + [3.0], device=env.device) - \
            torch.tensor([1.0] * 8 + [0.0], device=env.device)
        obs, rew, term, trunc, info = env.step(act)
        tobs, trew, tterm, ttrunc, _ = twin.step(act)
        for a, agent in enumerate(env.agents):
            fo, mask = info[agent]["final_observation"], info[agent]["_final_observation"]
            od = env.observation_space(agent).shape[0]
            if n == 1:
                assert isinstance(fo, np.ndarray) and fo.shape == (od,) and isinstance(mask, bool)
                if not bool(ever[0]):
                    assert rew[agent] == trew[agent] and term[agent] == tterm[agent] and trunc[agent] == ttrunc[agent]
                    if mask:
                        assert np.array_equal(fo, tobs[agent])
            else:
                assert fo.shape == (n, od) and mask.dtype == torch.bool and mask.shape == (n,)
                same = ~ever
                assert torch.equal(rew[agent][same], trew[agent][same]) and torch.equal(term[agent][same], tterm[agent][same])
                assert torch.equal(fo[mask & same], tobs[agent][mask & same])
                assert torch.equal(obs[agent][~mask & same], tobs[agent][~mask & same])
        ended = env.batch.term[:, 2].bool() | env.batch.trunc[:, 2].bool()
        ever |= ended
        assert bool((env.batch.timestep[ended] == 0).all())
        if t == 5:   # maxSteps 5: every env truncates on the sixth step
            assert bool(ended.all())
        else:
            assert not bool(env.batch.trunc[:, 2].bool().any())


@pytest.mark.gpu
def test_gpu_gymnasium_wrapper_passes_final_observation():
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL
    from mujoco_rl_environment_wrapper_b200.wrappers import GymnasiumWrapper
    env = MuJoCoRL({"xmlPath": os.path.join(LEVELS, "one_ant_arena.xml"), "agents": ["sender"], "maxSteps": 3, "autoReset": True})
    w = GymnasiumWrapper(env, "sender")
    w.reset()
    seen = []
    for _ in range(4):
        obs, rew, term, trunc, info = w.step(np.zeros(8, np.float32))
        seen.append(info["_final_observation"])
        assert info["final_observation"].shape == obs.shape
    assert seen == [False, False, False, True] and trunc


@pytest.mark.gpu
def test_gpu_refused_configurations():
    import torch
    from mujoco_rl_environment_wrapper_b200.batch import Batch

    def host_reward(env, agent):
        return 0.0
    with pytest.raises(Exception, match="autoReset"):
        _env(4, autoReset=True, rewardFunctions=[host_reward])
    with pytest.raises(Exception, match="autoReset"):
        _env(4, autoReset=True, xmlPath=[os.path.join(LEVELS, "two_ants.xml")] * 2)
    with pytest.raises(Exception, match="skipFrames"):
        _env(4, autoReset=True, skipFrames=0)
    env = _env(4, autoReset=True)
    with pytest.raises(Exception, match="step_host"):
        env.batch.step_host(*env.batch.host_arrays())
    model, spec, keep, low, high, A = scene_spec("2A", 10, 0.0, True)
    spec.flags |= L.SPEC_NO_PACK
    b = Batch(model, spec, 8, keepalive=keep)
    with pytest.raises(Exception, match="auto-reset"):
        b.set_subset(torch.arange(4, dtype=torch.int32))


@pytest.mark.gpu
def test_gpu_c2_rollout_65536_stays_finite():
    import torch
    env = _env(65536, autoReset=True, maxSteps=200)
    env.reset()
    ended = 0
    for _ in range(300):
        obs, rew, term, trunc, info = env.step(env.sample_actions())
        ended += int(info["sender"]["_final_observation"].sum())
    b = env.batch
    assert ended >= 65536
    assert bool(torch.isfinite(b.qpos).all() and torch.isfinite(b.qvel).all() and torch.isfinite(b.obs).all())
    assert bool(torch.isfinite(b.final_obs[:, :, :60]).all())
    assert int(b.ncon_dropped.sum()) == 0 and int(b.nreset.sum()) == 0
