"""Start states (DESIGN §5d): resets that start from caller-supplied rows (mjb_reset_rows, `reset(options=...)`) or from
a start-state pool drawn per reset in the kernel (mjb_env_spec.start_qpos / start_qvel / n_start, config
"startStates").  The kernel source runs on the host SIMT emulator in both lane orders, and through libmjb.so on the GPU:
- a one-row pool (qpos0, 0) changes nothing, bit for bit;
- a reset from rows equals the given rows (plus the documented noise), a forward pass on them and the observation
  gather, and leaves the other envs alone;
- pool resets and pool auto-resets equal: draw the row with a numpy restatement, write it, reset from rows."""
import ctypes
import os

import numpy as np
import pytest

import emu_harness as E
from common import LEVELS
from mujoco_rl_environment_wrapper_b200 import _lib as L
from test_autoreset import EmuSide, GpuSide, draw_u32_np, reset_action_np, reset_key_np, scene_spec

MODE_RESET_ROWS = 4   # csrc/env_kernel.cuh


def start_index_np(seed, env, ep, n_start):
    """include/mjb.h, mjb_start_index"""
    d = draw_u32_np(seed ^ 0x5EEDC0DE, env, 0xD000, ep).astype(np.uint64)
    return ((d * np.uint64(n_start)) >> np.uint64(32)).astype(np.int64)


def with_noise(model, seed, env, ep, noise, q, v):
    """start rows q [n, nq] / v [n, nv] of envs `env` with the reset_noise draws (keys `ep`) added, in float32 without
    fused multiply-add (as the host emulator evaluates them)"""
    if noise == 0.0:
        return q, v
    f = model.fields
    q, v = q.copy(), v.copy()
    u = lambda slot: (draw_u32_np(seed ^ 0x5EEDC0DE, env, slot, ep) >> np.uint32(8)).astype(np.float32) * np.float32(2.0 ** -24)
    for j in range(len(f["jnt_type"])):
        if int(f["jnt_type"][j]) != 0:   # not a free joint
            a = int(f["jnt_qposadr"][j])
            q[:, a] = q[:, a] + np.float32(noise) * (np.float32(2) * u(0x4000 + j) - np.float32(1))
    for j in range(model.nv):
        v[:, j] = v[:, j] + np.float32(noise) * (np.float32(2) * u(0x8000 + j) - np.float32(1))
    return q, v


class EmuRows(EmuSide):
    def __init__(self, model, spec, keep, n, skip_frames, reverse, pool=None):
        if pool is not None:
            self.pool = tuple(np.ascontiguousarray(x, np.float32) for x in pool)   # host memory: the emulator reads it
            spec.start_qpos, spec.start_qvel, spec.n_start = self.pool[0].ctypes.data, self.pool[1].ctypes.data, len(self.pool[0])
        super().__init__(model, spec, keep, n, skip_frames, reverse)

    def reset_rows(self, mask=None):
        self.eb.run(MODE_RESET_ROWS, mask=mask, reverse=self.reverse)

    def forward(self):
        self.eb.run(E.MODE_FORWARD, reverse=self.reverse)


class GpuRows(GpuSide):
    def __init__(self, model, spec, keep, n, skip_frames, reverse=False, pool=None):
        import torch
        from mujoco_rl_environment_wrapper_b200.batch import Batch
        ss = None if pool is None else tuple(torch.from_numpy(np.ascontiguousarray(x, np.float32)).cuda() for x in pool)
        self.b = Batch(model, spec, n, keepalive=keep, start_states=ss)
        if spec.flags & L.SPEC_AUTORESET:
            self.b.final_obs.fill_(float("nan"))

    def reset_rows(self, mask=None):
        import torch
        self.b.reset_rows(None if mask is None else torch.from_numpy(mask))

    def forward(self):
        self.b.forward()


def rollout_rows(side, model, scene, n, steps, seed, skip_frames=1, noise=0.0):
    """(qpos [n, nq], qvel [n, nv]) reached by `steps` random steps from reset (no episode ends on the way)"""
    m, spec, keep, low, high, A = scene_spec(scene, 10 ** 6, noise, False, seed + 1, skip_frames)
    if scene == "2A":
        spec.n_dones = 0
    s = side(m, spec, keep, n, skip_frames, False)
    s.reset()
    rng = np.random.default_rng(seed)
    for _ in range(steps):
        act = s.get("actions")
        act[:, :, :len(low)] = rng.uniform(low, high, (n, A, len(low))).astype(np.float32)
        s.put("actions", act)
        s.step()
    return s.get("qpos")[:, :model.nq].copy(), s.get("qvel")[:, :model.nv].copy()


def put_rows(side, env, qpos, qvel):
    q, v = side.get("qpos"), side.get("qvel")
    q[env, :qpos.shape[1]], v[env, :qvel.shape[1]] = qpos, qvel
    side.put("qpos", q)
    side.put("qvel", v)


def assert_same(a, b, tag, names=None):
    for k in names or b.names:
        assert a.get(k).tobytes() == b.get(k).tobytes(), (tag, k)


def random_actions(side, rng, low, high, A):
    act = side.get("actions")
    act[:, :, :len(low)] = rng.uniform(low, high, (act.shape[0], A, len(low))).astype(np.float32)
    return act


# ---- 1. a one-row pool (qpos0, 0) is today's reset ------------------------------------------------------------------
def run_neutral(side, scene, n, steps, noise, max_steps, skip_frames=1, reverse=False, seed=5):
    model, spec_p, keep_p, low, high, A = scene_spec(scene, max_steps, noise, True, seed, skip_frames)
    _, spec_r, keep_r, _, _, _ = scene_spec(scene, max_steps, noise, True, seed, skip_frames)
    pool = (np.float32(model.fields["qpos0"])[None, :model.nq], np.zeros((1, model.nv), np.float32))
    _, spec_b, keep_b, _, _, _ = scene_spec(scene, max_steps, noise, False, seed, skip_frames)
    pooled, plain = side(model, spec_p, keep_p, n, skip_frames, reverse, pool=pool), side(model, spec_r, keep_r, n, skip_frames, reverse)
    bare = side(model, spec_b, keep_b, n, skip_frames, reverse)   # no flag: the reset kernel batches without a pool run
    sides = (pooled, plain, bare)
    rng = np.random.default_rng(seed)
    e = np.arange(n)
    for s in sides:
        s.reset()
    assert_same(pooled, plain, "full reset")
    assert_same(pooled, bare, "full reset")
    for t in range(2):
        act = random_actions(plain, rng, low, high, A)
        for s in sides:
            s.put("actions", act)
            s.step()
    for k in bare.names:   # the batch without auto-reset did not restart the episodes the steps ended
        bare.put(k, plain.get(k))
    for s in sides:
        s.reset((e % 3 == 1).astype(np.uint8))
    assert_same(pooled, plain, "masked reset")
    assert_same(pooled, bare, "masked reset")
    sides = (pooled, plain)
    ts0 = ((e // 4 * 7 + e % 4) % max_steps).astype(np.int32)
    ended = 0
    for s in sides:
        s.put("timestep", ts0)
    for t in range(steps):
        act = random_actions(plain, rng, low, high, A)
        for s in sides:
            s.put("actions", act)
            s.step()
        assert_same(pooled, plain, ("auto-reset step", t), plain.names + ["final_obs"])
        ended += int((plain.get("term")[:, A] | plain.get("trunc")[:, A]).sum())
    return ended


@pytest.mark.parametrize("reverse", [False, True])
@pytest.mark.parametrize("noise", [0.0, 0.05])
@pytest.mark.parametrize("scene,n,steps,max_steps", [("2A", 8, 7, 5), ("S1", 8, 7, 4), ("C1", 6, 7, 4)])
def test_emulator_neutral_pool_is_todays_reset(scene, n, steps, max_steps, noise, reverse):
    assert run_neutral(EmuRows, scene, n, steps, noise, max_steps, reverse=reverse) >= n


# ---- 2. reset from the caller's rows ----------------------------------------------------------------------------------
def run_rows(side, scene, n, noise, skip_frames=1, reverse=False, seed=5):
    model, spec, keep, low, high, A = scene_spec(scene, 50, noise, False, seed, skip_frames)
    _, spec_f, keep_f, _, _, _ = scene_spec(scene, 50, 0.0, False, seed, skip_frames)
    nq, nv = model.nq, model.nv
    rq, rv = rollout_rows(side, model, scene, n, 6, seed, skip_frames)
    perm = np.roll(np.arange(n), 1)   # every env gets another env's state
    rq, rv = rq[perm], rv[perm]
    s = side(model, spec, keep, n, skip_frames, reverse)
    s.reset()
    rng = np.random.default_rng(seed + 2)
    for _ in range(3):
        s.put("actions", random_actions(s, rng, low, high, A))
        s.step()
    mask = (np.arange(n) % 3 != 0).astype(np.uint8)
    m = mask.astype(bool)
    env = np.nonzero(m)[0]
    put_rows(s, env, rq[m], rv[m])
    key = reset_key_np(s.get("timestep")[env], rq[m, 0], rv[m, 0])   # keyed by the caller's rows
    before = {k: s.get(k) for k in s.names}
    s.reset_rows(mask)
    after = {k: s.get(k) for k in s.names}
    for k in s.names:
        assert after[k][~m].tobytes() == before[k][~m].tobytes(), ("unmasked env changed", k)
    wq, wv = with_noise(model, seed, env, key, noise, rq[m], rv[m])
    # a free joint's quaternion is stored as the forward pass normalised it: equal to within rounding, the rest bit for bit
    quat = np.zeros(nq, bool)
    for j in range(len(model.fields["jnt_type"])):
        if int(model.fields["jnt_type"][j]) == 0:
            quat[int(model.fields["jnt_qposadr"][j]) + 3:int(model.fields["jnt_qposadr"][j]) + 7] = True
    assert np.abs(after["qpos"][m, :nq][:, quat] - wq[:, quat]).max(initial=0.0) < 1e-6
    got = after["qpos"][m, :nq].copy()
    got[:, quat] = wq[:, quat]
    assert got.tobytes() == wq.tobytes()
    assert after["qvel"][m, :nv].tobytes() == wv.tobytes()
    assert (after["timestep"][m] == 0).all() and not after["ctrl"][m].any()
    si = after["store_i"][m]
    assert (si[:, :, L.STORE_I["draws"]] == before["store_i"][m][:, :, L.STORE_I["draws"]]).all()
    si[:, :, L.STORE_I["draws"]] = 0
    assert not si.any() and not after["store_f"][m].any()
    assert not after["reward"][m].any() and not after["term"][m].any() and not after["trunc"][m].any()
    # observation columns gathered through obs_index (the plugin columns follow them)
    for a in range(A):
        for i in range(spec.obs_adr[a], spec.obs_adr[a + 1]):
            code = spec.obs_index[i]
            kind, adr = code >> 24, code & 0xFFFFFF
            src = (after["sensordata"], after["qpos"], after["qvel"])[kind][m, adr]
            assert after["obs"][m, a, i - spec.obs_adr[a]].tobytes() == src.tobytes(), (a, i)
    if noise == 0.0:
        # sensors, exported positions and the stored accelerations (next warm start) are a forward pass on the same rows
        # with ctrl and warm start zeroed (the other envs of a packed warp hold what they held in the reset launch)
        f = side(model, spec_f, keep_f, n, skip_frames, reverse)
        for k in s.names:
            f.put(k, before[k])
        for k in ("ctrl", "warmstart"):
            v = before[k].copy()
            v[m] = 0
            f.put(k, v)
        f.forward()
        for k in ("sensordata", "probe", "warmstart"):
            assert f.get(k)[m].tobytes() == after[k][m].tobytes(), k


@pytest.mark.parametrize("reverse", [False, True])
@pytest.mark.parametrize("noise", [0.0, 0.05])
@pytest.mark.parametrize("scene,n", [("2A", 8), ("S1", 8), ("C1", 6)])
def test_emulator_reset_from_rows(scene, n, noise, reverse):
    run_rows(EmuRows, scene, n, noise, reverse=reverse)


# ---- 3. pool draws equal "draw in numpy, write the row, reset from rows" ------------------------------------------------
def ref_pool_reset(ref, model, seed, env, pool, mask=None):
    """write pool rows drawn by the numpy restatement into the masked envs; set their timestep so that the reset_noise
    key of the written rows equals the key of the rows they replace (the reset sets timestep to 0 anyway)"""
    ts, q, v = ref.get("timestep"), ref.get("qpos"), ref.get("qvel")
    key = reset_key_np(ts[env], q[env, 0], v[env, 0])
    p = start_index_np(seed, env, key, len(pool[0]))
    put_rows(ref, env, pool[0][p], pool[1][p])
    ts2 = ref.get("timestep")
    ts2[env] = (reset_key_np(np.zeros(len(env), np.int32), pool[0][p, 0], pool[1][p, 0]) ^ key).view(np.int32)
    ref.put("timestep", ts2)
    return key, p


def run_pool(side, scene, n, steps, noise, max_steps, skip_frames=1, reverse=False, seed=5, P=7):
    model, spec_p, keep_p, low, high, A = scene_spec(scene, max_steps, noise, True, seed, skip_frames)
    _, spec_r, keep_r, _, _, _ = scene_spec(scene, max_steps, noise, False, seed, skip_frames)
    rq, rv = rollout_rows(side, model, scene, max(n, P) if side is EmuRows else n, 5, seed + 3, skip_frames)
    pool = (rq[:P], rv[:P])
    pooled, ref = side(model, spec_p, keep_p, n, skip_frames, reverse, pool=pool), side(model, spec_r, keep_r, n, skip_frames, reverse)
    rng = np.random.default_rng(seed)
    e = np.arange(n)
    used = set()
    # full reset: every env draws a row, keyed by the rows both batches start with
    pooled.reset()
    _, p = ref_pool_reset(ref, model, seed, e, pool)
    used |= set(p.tolist())
    ref.reset_rows()
    assert_same(pooled, ref, "full reset")
    for t in range(2):
        act = random_actions(ref, rng, low, high, A)
        for s in (pooled, ref):
            s.put("actions", act)
            s.step()
        ref_auto(ref, model, seed, low, high, A, pool, used)
        assert_same(pooled, ref, ("auto-reset step", t))
    mask = (e % 3 == 1).astype(np.uint8)
    pooled.reset(mask)
    _, p = ref_pool_reset(ref, model, seed, e[mask.astype(bool)], pool)
    used |= set(p.tolist())
    ref.reset_rows(mask)
    assert_same(pooled, ref, "masked reset")
    ts0 = ((e // 4 * 7 + e % 4) % max_steps).astype(np.int32)
    for s in (pooled, ref):
        s.put("timestep", ts0)
    ended = 0
    for t in range(steps):
        act = random_actions(ref, rng, low, high, A)
        for s in (pooled, ref):
            s.put("actions", act)
        before = pooled.get("final_obs")
        pooled.step()
        ref.step()
        fin, obs = ref_auto(ref, model, seed, low, high, A, pool, used)
        assert_same(pooled, ref, ("auto-reset step", t))
        fo = pooled.get("final_obs")
        assert fo[fin].tobytes() == obs[fin].tobytes() and fo[~fin].tobytes() == before[~fin].tobytes()
        ended += int(fin.sum())
    return ended, used


def ref_auto(ref, model, seed, low, high, A, pool, used):
    """after a plain step: the finished envs get the documented action, a drawn pool row and a reset from rows; then the
    step's reward / term / trunc are put back (test_autoreset.reference_step with the pool row written first)"""
    saved = {k: ref.get(k) for k in ("reward", "term", "trunc", "obs")}
    fin = (saved["term"][:, A] | saved["trunc"][:, A]).astype(bool)
    if fin.any():
        env = np.nonzero(fin)[0]
        acts = ref.get("actions")
        drawn = acts.copy()
        key, p = ref_pool_reset(ref, model, seed, env, pool)
        used |= set(p.tolist())
        for a in range(A):
            for d in range(len(low)):
                drawn[env, a, d] = reset_action_np(seed, env, a, d, key, low[d], high[d])
        ref.put("actions", drawn)
        ref.reset_rows(fin.astype(np.uint8))
        ref.put("actions", acts)
        for k in ("reward", "term", "trunc"):
            ref.put(k, saved[k])
    return fin, saved["obs"]


@pytest.mark.parametrize("reverse", [False, True])
@pytest.mark.parametrize("noise", [0.0, 0.05])
@pytest.mark.parametrize("scene,n,steps,max_steps", [("2A", 8, 7, 5), ("S1", 8, 7, 4), ("C1", 6, 7, 4)])
def test_emulator_pool_equals_drawn_rows(scene, n, steps, max_steps, noise, reverse):
    ended, used = run_pool(EmuRows, scene, n, steps, noise, max_steps, reverse=reverse)
    assert ended >= n and len(used) >= 3


# ---- 4. / 5. the exported draw, refusals, config validation (no GPU) ----------------------------------------------------
def test_start_index_export_matches_numpy_restatement():
    lib = L.load()
    rng = np.random.default_rng(4)
    for _ in range(300):
        seed, env, ep, P = int(rng.integers(0, 2 ** 63)), int(rng.integers(0, 1 << 20)), int(rng.integers(0, 2 ** 32)), \
            int(rng.choice([1, 2, 5, 1024, int(rng.integers(1, 2 ** 31))]))
        got = lib.mjb_start_index(seed, env, ep, P)
        assert got == int(start_index_np(seed, env, np.uint32(ep), P)) and 0 <= got < P
    assert lib.mjb_start_index(1, 2, 3, 0) == 0


def test_batch_create_refuses_bad_pool_without_gpu():
    model, spec, keep, low, high, A = scene_spec("2A", 10, 0.0, False)
    lib = L.load()
    h = ctypes.c_void_p()
    spec.n_start = -1
    assert lib.mjb_batch_create(model._h, ctypes.byref(spec), 4, 0, None, ctypes.byref(L.Buffers()), ctypes.byref(h)) == -2
    assert b"n_start" in lib.mjb_last_error()
    spec.n_start, spec.start_qpos, spec.start_qvel = 3, 16, None
    assert lib.mjb_batch_create(model._h, ctypes.byref(spec), 4, 0, None, ctypes.byref(L.Buffers()), ctypes.byref(h)) == -2
    assert b"start_qvel" in lib.mjb_last_error()


def test_start_states_config_validation_without_gpu():
    import torch
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import parse_start_states, state_rows
    cpu = torch.device("cpu")
    q, v = parse_start_states({"qpos": np.zeros((3, 5))}, 5, 4, cpu)
    assert q.shape == (3, 5) and v.shape == (3, 4) and q.dtype == torch.float32 and not v.any()
    q, v = parse_start_states({"qpos": torch.ones(2, 5), "qvel": np.ones((2, 4))}, 5, 4, cpu)
    assert v.shape == (2, 4) and bool(v.all())
    assert parse_start_states(None, 5, 4, cpu) is None
    for bad, msg in (({"qpos": np.zeros((3, 6))}, "expected shape"), ({"qpos": np.zeros((0, 5))}, "P >= 1"),
                     ({"qpos": np.zeros(5)}, "expected shape"), ({"qpos": np.zeros((2, 5)), "qvel": np.zeros((3, 4))}, "qvel"),
                     ({"qpos": np.full((2, 5), np.nan)}, "finite"), ({"qvel": np.zeros((2, 4))}, "startStates"), ([1, 2], "startStates")):
        with pytest.raises(Exception, match=msg):
            parse_start_states(bad, 5, 4, cpu)
    assert state_rows("x", np.zeros(5), 1, 5, cpu).shape == (1, 5)
    with pytest.raises(Exception, match="expected shape"):
        state_rows("x", np.zeros((3, 5)), 4, 5, cpu)


# ---- GPU ---------------------------------------------------------------------------------------------------------------
GPU_SCENES = [("2A", 30, 1), ("C1", 28, 1), ("1A", 26, 2), ("3S", 30, 5)]


@pytest.mark.gpu
@pytest.mark.parametrize("scene,max_steps,skip_frames", GPU_SCENES)
def test_gpu_neutral_pool_is_todays_reset(scene, max_steps, skip_frames):
    assert run_neutral(GpuRows, scene, 4096, 12, 0.05, max_steps, skip_frames) >= 1024


@pytest.mark.gpu
@pytest.mark.parametrize("scene,max_steps,skip_frames", GPU_SCENES)
def test_gpu_reset_from_rows(scene, max_steps, skip_frames):
    run_rows(GpuRows, scene, 4096, 0.0, skip_frames)


@pytest.mark.gpu
@pytest.mark.parametrize("scene,max_steps,skip_frames", GPU_SCENES)
def test_gpu_pool_equals_drawn_rows(scene, max_steps, skip_frames):
    ended, used = run_pool(GpuRows, scene, 4096, 20, 0.05 if scene in ("C1", "3S") else 0.0, max_steps, skip_frames, P=64)
    assert ended >= 1024 and len(used) >= 32


@pytest.mark.gpu
def test_gpu_reset_from_rolled_out_states_matches_oracle_forward():
    """after a reset from states a random rollout reached, qpos / qvel / sensordata match the fp64 oracle's forward pass"""
    from oracle import OracleSim
    from test_gpu_parity import RTOL, rel_err
    for scene, skip in (("2A", 1), ("C1", 1)):
        model, spec, keep, low, high, A = scene_spec(scene, 50, 0.0, False, 5, skip)
        n = 64
        rq, rv = rollout_rows(GpuRows, model, scene, n, 8, 9, skip)
        s = GpuRows(model, spec, keep, n, skip)
        s.reset()
        put_rows(s, np.arange(n), rq, rv)
        s.reset_rows()
        q, v, sd = s.get("qpos"), s.get("qvel"), s.get("sensordata")
        for e in range(0, n, 7):
            sim = OracleSim(model.blob)
            sim.qpos[:] = rq[e]
            sim.qvel[:] = rv[e]
            sim.ctrl[:] = 0
            sim.forward()
            assert rel_err(q[e, :model.nq], sim.qpos) < RTOL and rel_err(v[e, :model.nv], sim.qvel) < RTOL
            assert rel_err(sd[e, :model.nsensordata], sim.sensordata) < RTOL, (scene, e)


def _env(n, **kw):
    from mujoco_rl_environment_wrapper_b200 import plugins as P
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL
    cfg = {"xmlPath": os.path.join(LEVELS, "two_ants.xml"), "infoJson": os.path.join(LEVELS, "info_2A.json"),
           "agents": ["sender", "receiver"], "environmentDynamics": [P.Language], "rewardFunctions": [P.tag_distance_reward],
           "doneFunctions": [P.distance_done], "num_envs": n, "maxSteps": 5, "seed": 11}
    cfg.update(kw)
    return MuJoCoRL(cfg)


def _states(n, steps=6):
    """qpos / qvel rows of a random rollout of the 2A env (numpy [n, nq], [n, nv])"""
    env = _env(n, maxSteps=10 ** 6, doneFunctions=[])
    env.reset()
    for _ in range(steps):
        env.step(env.sample_actions())
    return env.batch.qpos[:, :env.model.nq].cpu().numpy(), env.batch.qvel[:, :env.model.nv].cpu().numpy()


@pytest.mark.gpu
def test_gpu_level_variants_with_pool(tmp_path):
    """every level's handle draws from the same pool; a pooled reset equals a reset from the drawn rows"""
    import torch
    from test_gpu_parity import _level_variants
    (xa, ja), (xb, jb) = _level_variants(tmp_path)
    n, P = 256, 16
    rq, rv = _states(P)
    kw = dict(xmlPath=[xa, xb], infoJson=[ja, jb], seed=7, maxSteps=50)
    pooled = _env(n, **kw, startStates={"qpos": rq, "qvel": rv})
    ref = _env(n, **kw)
    pooled.reset()
    b = ref.batch
    e = np.arange(n)
    key = reset_key_np(b.timestep.cpu().numpy(), b.qpos[:, 0].cpu().numpy(), b.qvel[:, 0].cpu().numpy())
    p = start_index_np(7, e, key, P)
    ref.reset(options={"qpos": torch.from_numpy(rq[p]).cuda(), "qvel": torch.from_numpy(rv[p]).cuda()})
    assert torch.equal(pooled.level_id, ref.level_id) and len(set(pooled.level_id.tolist())) == 2
    for k in ("qpos", "qvel", "obs", "sensordata", "reward", "term", "trunc", "store_i", "store_f", "timestep"):
        assert getattr(pooled.batch, k).cpu().numpy().tobytes() == getattr(b, k).cpu().numpy().tobytes(), k
    assert len(set(p.tolist())) >= 8


@pytest.mark.gpu
def test_gpu_reset_options_api():
    import torch
    # N = 1: numpy in, numpy out
    rq, rv = _states(4)
    env = _env(1)
    obs, _ = env.reset(options={"qpos": rq[2], "qvel": rv[2]})
    assert isinstance(obs["sender"], np.ndarray)
    # (qpos to within rounding: the forward pass stores free-joint quaternions normalised)
    assert np.allclose(env.batch.qpos[0, :env.model.nq].cpu().numpy(), rq[2], rtol=0, atol=1e-6)
    assert np.array_equal(env.batch.qvel[0, :env.model.nv].cpu().numpy(), rv[2])
    env.reset(options={"qpos": rq[1]})   # qvel defaults to zeros
    assert not env.batch.qvel[0].any()
    # N = 64: tensors, with and without mask
    n = 64
    rq, rv = _states(n)
    env = _env(n)
    env.reset()
    env.step(env.sample_actions())
    q_before = env.batch.qpos.clone()
    tq, tv = torch.from_numpy(rq).cuda(), torch.from_numpy(rv).cuda()
    mask = torch.arange(n, device=env.device) % 2 == 0
    obs, _ = env.reset(options={"qpos": tq, "qvel": tv}, mask=mask)
    nq, nv = env.model.nq, env.model.nv
    close = lambda a, b: torch.allclose(a, b, rtol=0, atol=1e-6)
    assert close(env.batch.qpos[mask, :nq], tq[mask]) and torch.equal(env.batch.qvel[mask, :nv], tv[mask])
    assert torch.equal(env.batch.qpos[~mask], q_before[~mask])
    assert bool((env.batch.timestep[mask] == 0).all()) and bool((env.batch.timestep[~mask] == 1).all())
    obs, _ = env.reset(options={"qpos": tq, "qvel": tv})
    assert close(env.batch.qpos[:, :nq], tq) and torch.equal(env.batch.qvel[:, :nv], tv)
    assert torch.is_tensor(obs["sender"]) and obs["sender"].shape[0] == n
    with pytest.raises(Exception, match="expected shape"):
        env.reset(options={"qpos": tq[:, :5]})
    with pytest.raises(Exception, match="expected shape"):
        _env(4, startStates={"qpos": rq[:, :7]})


@pytest.mark.gpu
def test_gpu_pool_with_autoreset_through_step():
    import torch
    n, P = 64, 8
    rq, rv = _states(P)
    env = _env(n, autoReset=True, startStates={"qpos": rq})
    env.reset()
    pool = torch.from_numpy(rq).cuda()
    is_start = lambda q: ((q[:, None, :env.model.nq] - pool[None]).abs() <= 1e-6).all(-1).any(-1)
    starts = is_start(env.batch.qpos)
    assert bool(starts.all()) and bool((env.batch.qvel == 0).all())
    ended = 0
    for t in range(12):
        obs, rew, term, trunc, info = env.step(env.sample_actions())
        fin = info["sender"]["_final_observation"]
        assert info["sender"]["final_observation"].shape == obs["sender"].shape
        if bool(fin.any()):   # the new episode starts from a pool row
            assert bool(is_start(env.batch.qpos[fin]).all()) and bool((env.batch.timestep[fin] == 0).all())
        ended += int(fin.sum())
    assert ended >= n


@pytest.mark.gpu
def test_gpu_gymnasium_wrapper_passes_options():
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL
    from mujoco_rl_environment_wrapper_b200.wrappers import GymnasiumWrapper
    env = MuJoCoRL({"xmlPath": os.path.join(LEVELS, "one_ant_arena.xml"), "agents": ["sender"], "maxSteps": 3})
    w = GymnasiumWrapper(env, "sender")
    o0, _ = w.reset()
    q = np.float32(env.model.fields["qpos0"])[:env.model.nq].copy()
    q[2] += 0.5
    o1, _ = w.reset(options={"qpos": q})
    assert np.allclose(env.batch.qpos[0, :env.model.nq].cpu().numpy(), q, rtol=0, atol=1e-6) and not np.array_equal(o0, o1)
    o2, _ = w.reset(options=None)
    assert np.array_equal(o2, o0)


@pytest.mark.gpu
def test_gpu_c2_rollout_65536_with_pool_stays_finite():
    import torch
    rq, rv = _states(1024, steps=10)
    env = _env(65536, autoReset=True, maxSteps=200, startStates={"qpos": rq, "qvel": rv})
    env.reset()
    ended = 0
    for _ in range(300):
        obs, rew, term, trunc, info = env.step(env.sample_actions())
        ended += int(info["sender"]["_final_observation"].sum())
    b = env.batch
    assert ended >= 65536
    assert bool(torch.isfinite(b.qpos).all() and torch.isfinite(b.qvel).all() and torch.isfinite(b.obs).all())
    assert int(b.ncon_dropped.sum()) == 0 and int(b.nreset.sum()) == 0
