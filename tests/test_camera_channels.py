"""Depth and segmentation images of the agent cameras, and the last frame of every episode an auto-reset step ends
(include/mjb.h, mjb_render_ex and mjb_env_spec.final_qpos).

Pinned here: an fp64 restatement of the ray caster's depth and segmentation (below), against closed forms and against
the oracle's RGB image of the same rays; on the emulator, the `final_qpos` rows an auto-reset step writes; on the GPU,
the CUDA channels against the restatement, the colour of `mjb_render_ex` against `mjb_render`, and the final frames
against a reference batch that renders before its masked reset."""
import ctypes
import os

import numpy as np
import pytest

from common import LEVELS
from mujoco_rl_environment_wrapper_b200 import _lib as L
from oracle.sim import OracleSim
from test_autoreset import EmuSide, GpuSide, reference_step, scene_spec

# the scene of test_cameras.py: a horizontal `front` camera 1 m above an infinite floor looking at a ball 4 m away
# (with an alpha-0 `ghost` sphere in between), a `down` camera 5 m above a crate, a tracking camera and an onboard one
SCENE = """<mujoco><compiler angle="degree"/><option timestep="0.002"/>
 <worldbody>
  <geom name="floor" type="plane" size="0 0 1" pos="0 0 0" rgba="0.2 0.6 0.4 1"/>
  <camera name="front" pos="0 0 1" xyaxes="0 -1 0 0 0 1" fovy="60"/>
  <camera name="down" pos="0 0 5" quat="1 0 0 0" fovy="40"/>
  <camera name="follow" mode="trackcom" pos="0 -3 0.3" xyaxes="1 0 0 0 0 1"/>
  <body name="ball" pos="4 0 1"><freejoint name="root"/><geom name="ball_geom" type="sphere" size="0.5" rgba="1 0 0.5 1"/>
   <camera name="onboard" pos="0 0 0.7" euler="90 0 0"/></body>
  <body name="crate" pos="0 0 0.25"><geom name="crate_geom" type="box" size="0.5 0.3 0.25" rgba="0 0 255 1"/></body>
  <body name="ghost" pos="2 0 1"><geom name="ghost_geom" type="sphere" size="0.4" rgba="1 1 1 0"/></body>
 </worldbody></mujoco>"""

PLANE, SPHERE, CAPSULE, BOX = 0, 2, 3, 6   # include/mjb_blob.h
MINVAL = 1e-15


# ---- fp64 restatement of the ray caster's depth and segmentation ---------------------------------------------------------
# The same rays and first-hit rule as csrc/render_kernel.cuh and the oracle's orc_render (the oracle's ray / geom tests,
# vectorised over the pixels); the kinematics come from the oracle.
def _quat_mat(q):
    w, x, y, z = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def _quad_roots(a, b, c):
    """roots of a x^2 + 2 b x + c = 0 (ascending) and where they exist"""
    det = b * b - a * c
    ok = (a >= MINVAL) & (det >= 0)
    with np.errstate(divide="ignore", invalid="ignore"):
        sq = np.sqrt(np.maximum(det, 0.0))
        a = np.where(ok, a, 1.0)
        return (-b - sq) / a, (-b + sq) / a, ok


def _first(best, t, ok):
    """keep the smaller non-negative t"""
    take = ok & (t >= 0) & ((best < 0) | (t < best))
    return np.where(take, t, best)


def _ray_geom(gtype, pos, R, size, o, d):
    """distance along the rays o + t d [P, 3] to the geom, -1 where missed"""
    lp, lv = R.T @ (o - pos), d @ R
    P = d.shape[0]
    if gtype == PLANE:
        with np.errstate(divide="ignore", invalid="ignore"):
            x = -lp[2] / lv[:, 2]
        p0, p1 = lp[0] + x * lv[:, 0], lp[1] + x * lv[:, 1]
        hit = (lv[:, 2] <= -MINVAL) & (x >= 0) & ((size[0] <= 0) | (np.abs(p0) <= size[0])) & \
            ((size[1] <= 0) | (np.abs(p1) <= size[1]))
        return np.where(hit, x, -1.0)
    if gtype == SPHERE:
        w = o - pos
        x0, x1, ok = _quad_roots(np.einsum("pi,pi->p", d, d), d @ w, np.full(P, w @ w - size[0] ** 2))
        return np.where(ok & (x0 >= 0), x0, np.where(ok & (x1 >= 0), x1, -1.0))
    best = np.full(P, -1.0)
    if gtype == CAPSULE:
        r, h = size[0], size[1]
        x0, x1, ok = _quad_roots(lv[:, 0] ** 2 + lv[:, 1] ** 2, lp[0] * lv[:, 0] + lp[1] * lv[:, 1],
                                 np.full(P, lp[0] ** 2 + lp[1] ** 2 - r * r))
        for x in (x0, x1):
            best = _first(best, x, ok & (np.abs(lp[2] + x * lv[:, 2]) <= h))
        for sg in (-1, 1):
            w = lp - np.array([0.0, 0.0, sg * h])
            x0, x1, ok = _quad_roots(np.einsum("pi,pi->p", lv, lv), lv @ w, np.full(P, w @ w - r * r))
            for x in (x0, x1):
                best = _first(best, x, ok & (sg * (lp[2] + x * lv[:, 2]) >= h))
        return best
    assert gtype == BOX
    for a in range(3):
        a1, a2 = (a + 1) % 3, (a + 2) % 3
        ok_a = np.abs(lv[:, a]) >= MINVAL
        for sg in (-1, 1):
            with np.errstate(divide="ignore", invalid="ignore"):
                t = (sg * size[a] - lp[a]) / lv[:, a]
            on = ok_a & (np.abs(lp[a1] + t * lv[:, a1]) <= size[a1]) & (np.abs(lp[a2] + t * lv[:, a2]) <= size[a2])
            best = _first(best, t, on)
    return best


def render_channels(sim, model, cam, width, height):
    """(depth f64 [H, W], segmentation i32 [H, W]) of fixed camera `cam` at the oracle's current kinematic state (call
    sim.forward() first); rows bottom-up.  Depth: hit distance along the optical axis (-z of the camera), 0 where nothing
    is hit; segmentation: the hit's geom id, -1 where nothing is hit; alpha-0 geoms are invisible."""
    f = model.fields
    if f["cam_mode"][cam] != 0:
        raise ValueError(f"camera {cam} cannot be rendered")
    b = int(f["cam_bodyid"][cam])
    xmat = sim.xmat[b].reshape(3, 3)
    o = sim.xpos[b] + xmat @ f["cam_pos"][3 * cam:3 * cam + 3]
    R = xmat @ _quat_mat(f["cam_quat"][4 * cam:4 * cam + 4])
    th = np.tan(0.5 * f["cam_fovy"][cam] * np.pi / 180.0)
    iy, ix = np.meshgrid(np.arange(height), np.arange(width), indexing="ij")
    dl = np.stack([((ix + 0.5) / width * 2 - 1) * th * (width / height), ((iy + 0.5) / height * 2 - 1) * th,
                   -np.ones(ix.shape)], axis=-1).reshape(-1, 3)
    norm = np.linalg.norm(dl, axis=1)
    d = (dl / norm[:, None]) @ R.T
    best, seg = np.full(len(d), np.inf), np.full(len(d), -1, np.int32)
    for g in range(model.ngeom):
        if f["geom_rgba"][4 * g + 3] <= 0:
            continue
        t = _ray_geom(int(f["geom_type"][g]), sim.geom_xpos[g], sim.geom_xmat[g].reshape(3, 3), f["geom_size"][3 * g:3 * g + 3], o, d)
        take = (t >= 0) & (t < best)
        best[take], seg[take] = t[take], g
    depth = np.where(seg >= 0, best / norm, 0.0)
    return depth.reshape(height, width), seg.reshape(height, width)


# ---- the restatement against closed forms and the oracle's colour image ----------------------------------------------------
def test_restated_depth_and_segmentation_closed_forms():
    m = L.Model(SCENE)
    s = OracleSim(m.blob)
    s.reset()
    s.forward()
    W = H = 128
    ball, crate, ghost, floor = (m.name2id(L.OBJ_GEOM, n) for n in ("ball_geom", "crate_geom", "ghost_geom", "floor"))
    th = np.tan(np.radians(30))
    depth, seg = render_channels(s, m, 0, W, H)
    rgb = s.render(0, W, H).astype(int)
    # the ball straight ahead: 4 m to its centre, radius 0.5 -> 3.5 m on the axis.  The centre pixel's ray is half a pixel
    # off the axis in u and v (angle a): it meets the sphere at t = 4 cos a - sqrt(0.25 - 16 sin^2 a), depth t cos a
    uv = 0.5 / (W / 2) * th
    ca = 1.0 / np.sqrt(1 + 2 * uv * uv)
    t = 4 * ca - np.sqrt(0.25 - 16 * (1 - ca * ca))
    assert seg[H // 2, W // 2] == ball and abs(depth[H // 2, W // 2] - t * ca) < 1e-12 and abs(t * ca - 3.5) < 1e-3
    # the ball's pixels are those the oracle paints in its colour, and the alpha-0 ghost in front of it never appears
    assert np.array_equal(seg == ball, (rgb[:, :, 0] > 100) & (rgb[:, :, 1] == 0))
    assert not (seg == ghost).any()
    # floor pixels of column 5 below the horizon: the camera is 1 m up, so depth = 1 / (|v| tan 30) with v the row's
    # image-plane coordinate
    rows = np.arange(H // 2)
    assert (seg[rows, 5] == floor).all()
    want = 1.0 / (np.abs(2 * (rows + 0.5) / H - 1) * th)
    assert np.allclose(depth[rows, 5], want, rtol=1e-12, atol=0)
    # above the horizon, away from the ball: nothing
    assert (depth[H // 2:, 5] == 0).all() and (seg[H // 2:, 5] == -1).all()
    # looking straight down onto the crate's top face 4.5 m below, and the floor 5 m below
    d_down, s_down = render_channels(s, m, 1, W, H)
    assert (s_down == crate).sum() > 100 and (s_down == floor).sum() > 100 and set(np.unique(s_down)) == {crate, floor}
    assert np.allclose(d_down[s_down == crate], 4.5, rtol=0, atol=1e-12)
    assert np.allclose(d_down[s_down == floor], 5.0, rtol=0, atol=1e-12)
    assert np.array_equal(s_down == crate, s.render(1, W, H)[:, :, 2] > 250)
    # tracking cameras are refused
    with pytest.raises(ValueError):
        render_channels(s, m, 2, 8, 8)


@pytest.mark.parametrize("level,cams", [("scene", (0, 1, 3)), ("two_ants_cams.xml", (0, 1))])
def test_restated_hits_are_the_oracles(level, cams):
    """segmentation -1 exactly where depth is 0 and exactly where the oracle's image is black, on the test scene and on
    the two-ant camera level after an oracle rollout (capsules, boxes, the finite floor)"""
    m = L.Model(SCENE if level == "scene" else open(os.path.join(LEVELS, level)).read())
    s = OracleSim(m.blob)
    s.reset()
    rng = np.random.default_rng(2)
    for _ in range(0 if level == "scene" else 150):
        s.ctrl[:] = rng.uniform(-1, 1, m.nu)
        s.step()
    s.forward()
    seen = set()
    for cam in cams:
        for W, H in ((48, 32), (30, 20)):
            depth, seg = render_channels(s, m, cam, W, H)
            assert np.array_equal(seg < 0, depth == 0) and (depth >= 0).all()
            black = s.render(cam, W, H).sum(axis=2) == 0
            assert np.array_equal(seg < 0, black), (cam, W, H)
            seen |= set(np.unique(seg).tolist())
    assert len(seen - {-1}) >= 3


# ---- final_qpos on the emulator -----------------------------------------------------------------------------------------
class _Capture:
    """a side for test_autoreset.reference_step that remembers the qpos rows of every plain step, before any reset"""
    def step(self):
        super().step()
        self.stepped_qpos = self.get("qpos")


class EmuRef(_Capture, EmuSide):
    pass


class EmuFinal(EmuSide):
    """auto-reset emulator batch with a sentinel-filled final_qpos buffer"""
    def __init__(self, model, spec, keep, n, skip_frames, reverse):
        super().__init__(model, spec, keep, n, skip_frames, reverse)
        self.final_qpos = np.full_like(self.eb.qpos, np.nan)
        spec.final_qpos = self.final_qpos.ctypes.data

    def get(self, k):
        return self.final_qpos.copy() if k == "final_qpos" else super().get(k)


def final_qpos_against_reference(auto_cls, ref_cls, scene, n, steps, max_steps, noise, reverse=False, seed=5):
    """auto-reset batch with final_qpos beside test_autoreset's reference path; every step: every buffer equal, the
    finished envs' final_qpos rows equal the reference's rows after its plain step, the other rows untouched"""
    model, spec_a, keep_a, low, high, A = scene_spec(scene, max_steps, noise, True, seed)
    _, spec_r, keep_r, _, _, _ = scene_spec(scene, max_steps, noise, False, seed)
    auto, ref = auto_cls(model, spec_a, keep_a, n, 1, reverse), ref_cls(model, spec_r, keep_r, n, 1, reverse)
    rng = np.random.default_rng(seed)
    e = np.arange(n)
    ts0 = ((e // 4 * 7 + e % 4) % max_steps).astype(np.int32)   # resets hit some copies of a packed warp and not others
    for s in (auto, ref):
        s.reset()
        s.put("timestep", ts0)
    nq, ever = model.nq, np.zeros(n, bool)
    for t in range(steps):
        act = auto.get("actions")
        act[:, :, :len(low)] = rng.uniform(low, high, (n, A, len(low))).astype(np.float32)
        for s in (auto, ref):
            s.put("actions", act)
        before = auto.get("final_qpos")
        auto.step()
        fin, _ = reference_step(ref, seed, low, high, A)
        for k in ref.names:
            assert auto.get(k).tobytes() == ref.get(k).tobytes(), (scene, t, k)
        fq = auto.get("final_qpos")
        assert fq[fin, :nq].tobytes() == ref.stepped_qpos[fin, :nq].tobytes(), (scene, t)
        assert fq[~fin].tobytes() == before[~fin].tobytes(), (scene, t)
        assert np.isnan(fq[:, nq:]).all()   # the row padding is never written
        ever |= fin
    return ever


@pytest.mark.parametrize("reverse", [False, True])
@pytest.mark.parametrize("noise", [0.0, 0.05])
@pytest.mark.parametrize("scene,n,steps,max_steps", [("2A", 8, 7, 5), ("S1", 8, 7, 4), ("C1", 6, 6, 4)])
def test_emulator_final_qpos_is_the_finishing_state(scene, n, steps, max_steps, noise, reverse):
    ever = final_qpos_against_reference(EmuFinal, EmuRef, scene, n, steps, max_steps, noise, reverse)
    assert ever.all()


# ---- refusals that need no device ------------------------------------------------------------------------------------------
def test_render_ex_refuses_without_a_batch():
    lib = L.load()
    a = L.RenderArgs()
    assert lib.mjb_render_ex(None, ctypes.byref(a)) == -2
    assert b"null" in lib.mjb_last_error()


def test_final_images_need_autoreset():
    """checked before any device work (the object is not constructed: that needs a GPU)"""
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL
    env = MuJoCoRL.__new__(MuJoCoRL)
    env.agent_cameras, env.auto_reset = True, False
    with pytest.raises(Exception, match="autoReset"):
        env.get_camera_images("sender", final=True)
    env.agent_cameras = False
    with pytest.raises(Exception, match="agentCameras"):
        env.get_camera_images("sender")


# ---- GPU ---------------------------------------------------------------------------------------------------------------
def _cams_batch(n, **kw):
    from common import make_spec
    from mujoco_rl_environment_wrapper_b200.batch import Batch
    from mujoco_rl_environment_wrapper_b200.tables import Tables
    text = open(os.path.join(LEVELS, "two_ants_cams.xml")).read()
    model = L.Model(text)
    tables = Tables(text, model, ["sender", "receiver"], False)
    spec, keep = make_spec(model, tables, ["sender", "receiver"], False)
    return model, spec, Batch(model, spec, n, keepalive=keep, **kw)


CHANNELS = [dict(rgb=r, depth=d, segmentation=s) for r in (True, False) for d in (True, False) for s in (True, False)
            if r or d or s]


@pytest.mark.gpu
def test_gpu_channels_match_restatement_and_rgb_is_unchanged():
    import torch
    model, spec, b = _cams_batch(24)
    N = 24
    b.reset()
    g = torch.Generator(device="cuda").manual_seed(5)
    for _ in range(120):   # the ants fall, flail and turn: the cameras see floor, walls, boxes and each other
        b.actions[:, :, :spec.n_phys_act] = torch.rand((N, 2, spec.n_phys_act), generator=g, device="cuda") * 2 - 1
        b.step()
    qpos = b.qpos.cpu().numpy()
    sim = OracleSim(model.blob)
    for W, H in ((64, 64), (30, 20)):
        rgb = b.render([0, 1], W, H)
        full = b.render_ex([0, 1], W, H, depth=True, segmentation=True)
        for ch in CHANNELS:   # the colour is mjb_render's, and no channel depends on which others are requested
            out = b.render_ex([0, 1], W, H, **ch)
            assert set(out) == {k for k, v in ch.items() if v}
            for k, v in out.items():
                assert torch.equal(v, rgb if k == "rgb" else full[k]), (W, H, ch, k)
        depth, seg = full["depth"].cpu().numpy(), full["segmentation"].cpu().numpy()
        assert depth.dtype == np.float32 and seg.dtype == np.int32 and depth.shape == seg.shape == (N, 2, H, W)
        assert np.array_equal(seg < 0, depth == 0)
        agree = total = 0
        worst = 0.0
        for e in range(N):
            sim.array("qpos")[:] = qpos[e, :model.nq]
            sim.forward()
            for k in range(2):
                rd, rs = render_channels(sim, model, k, W, H)
                same = seg[e, k] == rs
                agree += int(same.sum())
                total += same.size
                hit = same & (rs >= 0)
                rel = np.abs(depth[e, k][hit] - rd[hit]) / rd[hit]
                worst = max(worst, float(rel.max(initial=0.0)))
        assert agree / total >= 0.995, f"segmentation agrees on {agree} of {total} pixels"
        assert worst <= 1e-4, worst
        assert len(np.unique(seg)) >= 4
    with pytest.raises(Exception, match="camera id"):
        b.render_ex([5], 8, 8, depth=True)


@pytest.mark.gpu
def test_gpu_render_ex_refusals():
    import torch
    model, spec, b = _cams_batch(4)
    lib = L.load()
    b.reset()
    ids = (ctypes.c_int32 * 1)(0)

    def call(**kw):
        a = L.RenderArgs()
        a.cam_ids, a.ncams, a.width, a.height = ctypes.cast(ids, ctypes.POINTER(ctypes.c_int32)), 1, 8, 8
        for k, v in kw.items():
            setattr(a, k, v)
        return lib.mjb_render_ex(b._h, ctypes.byref(a)), lib.mjb_last_error()
    depth = torch.zeros((4, 1, 8, 8), device="cuda")
    assert call(depth=depth.data_ptr())[0] == 0
    rc, msg = call()
    assert rc == -2 and b"all NULL" in msg
    rc, msg = call(depth=depth.data_ptr(), width=0)
    assert rc == -2 and b"pixels" in msg
    rc, msg = call(depth=depth.data_ptr(), ncams=9)
    assert rc == -2 and b"cameras" in msg
    other = torch.zeros_like(b.qpos)
    rc, msg = call(depth=depth.data_ptr(), qpos=other.data_ptr())   # neither the batch's qpos nor a final_qpos
    assert rc == -2 and b"final_qpos" in msg
    assert call(depth=depth.data_ptr(), qpos=b.qpos.data_ptr())[0] == 0
    with pytest.raises(Exception, match="final_qpos"):
        b.render_ex([0], 8, 8, final=True)


def _cams_env(n, **kw):
    from mujoco_rl_environment_wrapper_b200 import plugins as P
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL
    cfg = {"xmlPath": os.path.join(LEVELS, "two_ants_cams.xml"), "agents": ["sender", "receiver"], "agentCameras": True,
           "environmentDynamics": [P.Language], "num_envs": n, "maxSteps": 30, "seed": 11, "resetNoise": 0.05,
           "sensorResolution": (32, 24)}
    cfg.update(kw)
    return MuJoCoRL(cfg)


class _EnvRef(GpuSide):
    """a MuJoCoRL twin without autoReset, driven through its batch for test_autoreset.reference_step: every plain step
    renders all three channels of both agent cameras before the masked reset"""
    def __init__(self, env):
        self.env, self.b = env, env.batch

    def step(self):
        self.b.step()
        self.images = self.env.get_camera_images("sender") | {"all": self.b.render_ex([0, 1], 32, 24, depth=True, segmentation=True)}


@pytest.mark.gpu
def test_gpu_final_frames_equal_the_frames_before_the_reset():
    import torch
    N, A = 4096, 2
    auto, twin = _cams_env(N, autoReset=True), _cams_env(N)
    assert getattr(twin.batch, "final_qpos", None) is None and auto.batch.final_qpos.shape == (N, auto.batch.layout.qpos_stride)
    ref = _EnvRef(twin)
    e = torch.arange(N, device="cuda")
    ts0 = ((e // 4 * 7 + e % 4) % 30).to(torch.int32)   # staggered episodes: about N / 30 end on every step
    for env in (auto, twin):
        env.reset()
        env.batch.timestep.copy_(ts0)
    asp = auto.action_space("sender")
    low, high = np.asarray(asp.low, np.float32), np.asarray(asp.high, np.float32)
    g = torch.Generator(device="cuda").manual_seed(3)
    ended = 0
    for t in range(36):
        act = torch.rand((N, A, len(low)), generator=g, device="cuda") * torch.tensor(high - low, device="cuda") + \
            torch.tensor(low, device="cuda")
        auto.step(act)
        twin.batch.actions[:, :, :len(low)] = act
        fin, _ = reference_step(ref, 11, low, high, A)
        fin_t = torch.from_numpy(fin).cuda()
        for k in ("qpos", "qvel", "obs", "timestep", "store_i"):   # lock-step
            assert torch.equal(auto.batch.buf[k], twin.batch.buf[k]), (t, k)
        got = auto.get_camera_images("sender", final=True)
        assert torch.equal(got["mask"], fin_t)
        for k in ("rgb", "depth", "segmentation"):
            want = ref.images[k]
            assert torch.equal(got[k][fin_t], want[fin_t]), (t, k)
            assert not got[k][~fin_t].any(), (t, k)
        # Batch level: all cameras, and envs outside the mask keep what the output held
        sentinel = {"rgb": torch.full((N, 2, 24, 32, 3), 7, dtype=torch.uint8, device="cuda"),
                    "depth": torch.full((N, 2, 24, 32), -3.0, device="cuda"),
                    "segmentation": torch.full((N, 2, 24, 32), -9, dtype=torch.int32, device="cuda")}
        keep = {k: v.clone() for k, v in sentinel.items()}
        out = auto.batch.render_ex([0, 1], 32, 24, depth=True, segmentation=True, final=True, mask=fin_t, out=sentinel)
        for k in keep:
            assert torch.equal(out[k][fin_t], ref.images["all"][k][fin_t]), (t, k)
            assert torch.equal(out[k][~fin_t], keep[k][~fin_t]), (t, k)
        ended += int(fin.sum())
    assert ended >= N


class _GpuFinal(GpuSide):
    def __init__(self, model, spec, keep, n, skip_frames, reverse=False):
        from mujoco_rl_environment_wrapper_b200.batch import Batch
        self.b = Batch(model, spec, n, keepalive=keep, final_qpos=True)
        self.b.final_obs.fill_(float("nan"))
        self.b.final_qpos.fill_(float("nan"))

    def get(self, k):
        return self.b.final_qpos.cpu().numpy().copy() if k == "final_qpos" else super().get(k)


class _GpuRef(_Capture, GpuSide):
    pass


@pytest.mark.gpu
@pytest.mark.parametrize("scene,max_steps", [("2A", 30), ("C1", 28)])
def test_gpu_final_qpos_is_the_finishing_state(scene, max_steps):
    ever = final_qpos_against_reference(_GpuFinal, _GpuRef, scene, 4096, 20, max_steps, 0.05)
    assert ever.sum() >= 4096 // 2


@pytest.mark.gpu
@pytest.mark.parametrize("scene,max_steps", [("2A", 30), ("C1", 28)])
def test_gpu_specialised_and_generic_final_qpos_agree(scene, max_steps):
    import torch
    n = 4096
    model, spec, keep, low, high, A = scene_spec(scene, max_steps, 0.05, True)
    _, gspec, gkeep, _, _, _ = scene_spec(scene, max_steps, 0.05, True)
    gspec.flags |= L.SPEC_GENERIC
    sides = [_GpuFinal(model, spec, keep, n, 1), _GpuFinal(model, gspec, gkeep, n, 1)]
    assert sides[0].b.geometry()["specialised"] and not sides[1].b.geometry()["specialised"]
    ts0 = (np.arange(n) % max_steps).astype(np.int32)
    for s in sides:
        s.reset()
        s.put("timestep", ts0)
    rng = np.random.default_rng(1)
    for t in range(2 * max_steps):
        act = sides[0].get("actions")
        act[:, :, :len(low)] = rng.uniform(low, high, (n, A, len(low))).astype(np.float32)
        for s in sides:
            s.put("actions", act)
            s.step()
        for k in ("final_qpos", "qpos", "final_obs"):
            assert sides[0].get(k).tobytes() == sides[1].get(k).tobytes(), (scene, t, k)
    assert not np.isnan(sides[0].get("final_qpos")[:, :model.nq]).any()   # every env ended an episode
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_gpu_single_env_shapes_follow_get_camera_data():
    env = _cams_env(1, sensorResolution=(64, 64))
    env.reset()
    env.step(env.sample_actions())
    for cam, shape in (("sender", (1, 64, 64)), ("receiver_camera", (64, 64))):
        out = env.get_camera_images(cam)
        rgb = env.get_camera_data(cam)
        assert set(out) == {"rgb", "depth", "segmentation"}
        assert isinstance(out["rgb"], np.ndarray) and out["rgb"].dtype == rgb.dtype and out["rgb"].shape == rgb.shape == shape + (3,)
        assert np.array_equal(out["rgb"], rgb)
        assert isinstance(out["depth"], np.ndarray) and out["depth"].dtype == np.float32 and out["depth"].shape == shape
        assert isinstance(out["segmentation"], np.ndarray) and out["segmentation"].dtype == np.int32 and out["segmentation"].shape == shape
    assert set(env.get_camera_images("sender", depth=False, segmentation=False)) == {"rgb"}
    with pytest.raises(Exception, match="autoReset"):
        env.get_camera_images("sender", final=True)
    auto = _cams_env(1, autoReset=True, maxSteps=2, sensorResolution=(64, 64))
    auto.reset()
    masks = []
    for _ in range(3):
        auto.step(auto.sample_actions())
        out = auto.get_camera_images("sender", final=True)
        masks.append(out["mask"])
        assert isinstance(out["mask"], bool) and out["rgb"].shape == (1, 64, 64, 3)
        assert out["rgb"].any() == out["mask"]
    assert masks == [False, False, True]
    many = _cams_env(6, sensorResolution=(32, 32))
    many.reset()
    out = many.get_camera_images("sender")
    assert tuple(out["rgb"].shape) == (6, 1, 32, 32, 3) and tuple(out["depth"].shape) == (6, 1, 32, 32)
    assert bool((out["rgb"] == many.get_camera_data("sender")).all())
    with pytest.raises(KeyError):
        many.get_camera_images("no_such_camera")
