"""Per-env physical parameters (DESIGN §5e): a table `params [N, n_params]` of body masses / inertias, geom frictions,
actuator gears and dof dampings (mjb_env_spec.params, config "perEnvParams"), optionally redrawn at every reset
(MJB_SPEC_RANDOMIZE, config "randomizeParams").  The reference for "an env whose row holds V" is a batch of the model
blob with the five fields (and the pairs' mixed friction) patched to V, stored as fp64 copies of the fp32 values.  The
kernel source runs on the host SIMT emulator in both lane orders, and through libmjb.so on the GPU:
- a table of nominal rows changes nothing, bit for bit (models without any damping: within the §3d tolerance, since
  the table kernels always take the implicit-damping path);
- an env with its own row equals that env of the patched-blob batch;
- randomising resets and auto-resets equal: draw the scales in numpy, write the rows, reset without randomisation."""
import ctypes
import os
import struct
import subprocess
import tempfile

import numpy as np
import pytest

import emu_harness as E
from common import LEVELS, load_scene
from mujoco_rl_environment_wrapper_b200 import _lib as L
from test_autoreset import EmuSide, GpuSide, draw_u32_np, reset_action_np, reset_key_np, scene_spec

_HERE = os.path.dirname(os.path.abspath(__file__))
_EMU = None
MODE_RESET_ROWS = 4   # csrc/env_kernel.cuh


def emu_params_lib():
    """tests/emu/emu_params.cpp built into a temporary directory (the kernels with PRM)"""
    global _EMU
    if _EMU is None:
        so = os.path.join(tempfile.mkdtemp(prefix="mjb_emu_params_"), "libmjb_emu_params.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", so,
                               os.path.join(_HERE, "emu", "emu_params.cpp")])
        lib = ctypes.CDLL(so)
        lib.emu_last_error.restype = ctypes.c_char_p
        lib.emu_param_spec_error.restype = ctypes.c_char_p
        lib.emu_param_spec_error.argtypes = [ctypes.POINTER(L.EnvSpec)]
        lib.emu_run.argtypes = [ctypes.c_char_p, ctypes.POINTER(L.EnvSpec), ctypes.c_int, ctypes.POINTER(L.Buffers),
                                ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
        _EMU = lib
    return _EMU


# ---- numpy restatements ------------------------------------------------------------------------------------------------
def param_scale_np(seed, env, family, index, ep, lo, hi):
    """include/mjb.h, mjb_param_scale (float32, no fused multiply-add)"""
    u = (draw_u32_np(seed ^ 0x5EEDC0DE, env, 0x10000 + 0x1000 * family + np.asarray(index, np.uint64), ep) >> np.uint32(8)).astype(np.float32) \
        * np.float32(2.0 ** -24)
    return np.float32(lo) + u * (np.float32(hi) - np.float32(lo))


def kernel_bodies(model):
    """bodies the kernel simulates (below a joint somewhere on their chain); the table's other body entries are ignored"""
    f = model.fields
    moving = np.zeros(model.nbody, bool)
    for b in range(1, model.nbody):
        moving[b] = f["body_dofnum"][b] > 0 or moving[f["body_parentid"][b]]
    return moving


def drawn_rows(model, rows, seed, env, ep, ranges):
    """rows [len(env), n_params] after a randomising reset of envs `env` with keys `ep`: nominal * s on every entry the
    kernel uses (family 0's s is the body's, for its mass and its three inertia entries)"""
    lay, nom = model.param_layout(), model.nominal_params()
    out = rows.copy()
    env, ep = np.asarray(env), np.asarray(ep)
    fam = [("body_mass", 0, 1), ("body_inertia", 0, 3), ("geom_friction", 1, 1), ("actuator_gear", 2, 1), ("dof_damping", 3, 1)]
    count = {"body_mass": model.nbody, "body_inertia": model.nbody, "geom_friction": model.ngeom, "actuator_gear": model.nu,
             "dof_damping": model.nv}
    moving = kernel_bodies(model)
    for name, f, w in fam:
        o = getattr(lay, name)
        for i in range(count[name]):
            if f == 0 and not moving[i]:
                continue
            s = param_scale_np(seed, env, f, i, ep, *ranges[f])
            for j in range(w):
                out[:, o + w * i + j] = np.float32(nom[o + w * i + j]) * s
    return out


def blob_offsets(raw):
    _, nf, _, _ = struct.unpack_from("8siiq", raw, 0)
    out = {}
    for i in range(nf):
        name, dt, cnt, off = struct.unpack_from("32siiq", raw, 24 + i * 48)
        out[name.split(b"\0")[0].decode()] = (dt, cnt, off)
    return out


def patched_blob(model, row):
    """the model blob with its five fields replaced by `row` (fp64 copies of the fp32 values) and every collision pair's
    sliding friction the max of its two geoms'; *_invweight0 stay nominal"""
    raw = bytearray(model.blob)
    offs, f, lay = blob_offsets(bytes(raw)), model.fields, model.param_layout()
    row = np.asarray(row, np.float32).astype(np.float64)

    def put(name, idx, vals):
        dt, cnt, off = offs[name]
        a = np.frombuffer(raw, np.float64, cnt, off).copy()
        a[idx] = vals
        raw[off:off + 8 * cnt] = a.tobytes()
    nb, ng = model.nbody, model.ngeom
    put("body_mass", slice(None), row[lay.body_mass:lay.body_mass + nb])
    put("body_inertia", slice(None), row[lay.body_inertia:lay.body_inertia + 3 * nb])
    fr = row[lay.geom_friction:lay.geom_friction + ng]
    put("geom_friction", slice(0, None, 3), fr)
    put("actuator_gear", slice(None), row[lay.actuator_gear:lay.actuator_gear + model.nu])
    put("dof_damping", slice(None), row[lay.dof_damping:lay.dof_damping + model.nv])
    if f["pair_geom1"].size:
        put("pair_friction", slice(0, None, 3), np.maximum(fr[f["pair_geom1"]], fr[f["pair_geom2"]]))
    return bytes(raw)


class _BlobModel:
    """a model whose blob was patched: what EmuBatch needs of it"""
    def __init__(self, model, blob):
        self.blob, self._m = blob, model

    def __getattr__(self, k):
        return getattr(self._m, k)


# ---- emulator / GPU sides with a table ---------------------------------------------------------------------------------
class EmuPrm(EmuSide):
    def __init__(self, model, spec, keep, n, skip_frames, reverse, table=False, ranges=None):
        self.params = None
        if table or ranges is not None:
            self.params = np.ascontiguousarray(np.tile(model.nominal_params(), (n, 1)), np.float32)
            spec.params = self.params.ctypes.data
            if ranges is not None:
                spec.flags |= L.SPEC_RANDOMIZE
                for f, (lo, hi) in enumerate(ranges):
                    spec.param_lo[f], spec.param_hi[f] = lo, hi
        super().__init__(model, spec, keep, n, skip_frames, reverse)
        self.eb.lib = emu_params_lib()

    names = property(lambda self: list(self.eb.buf) + (["params"] if self.params is not None else []))

    def forward(self):
        self.eb.run(E.MODE_FORWARD, reverse=self.reverse)

    def reset_rows(self, mask=None):
        self.eb.run(MODE_RESET_ROWS, mask=mask, reverse=self.reverse)

    def get(self, k):
        return self.params.copy() if k == "params" else super().get(k)

    def put(self, k, v):
        if k == "params":
            self.params[...] = v
        else:
            super().put(k, v)


class GpuPrm(GpuSide):
    def __init__(self, model, spec, keep, n, skip_frames, reverse=False, table=False, ranges=None):
        from mujoco_rl_environment_wrapper_b200.batch import Batch
        self.b = Batch(model, spec, n, keepalive=keep, params=table, param_ranges=ranges)
        self.params = getattr(self.b, "params", None)
        if spec.flags & L.SPEC_AUTORESET:
            self.b.final_obs.fill_(float("nan"))

    names = property(lambda self: list(self.b.buf) + (["params"] if self.params is not None else []))

    def forward(self):
        self.b.forward()

    def reset_rows(self, mask=None):
        import torch
        self.b.reset_rows(None if mask is None else torch.from_numpy(mask))

    def get(self, k):
        return self.params.cpu().numpy().copy() if k == "params" else super().get(k)

    def put(self, k, v):
        import torch
        if k == "params":
            self.params.copy_(torch.from_numpy(np.ascontiguousarray(v)))
        else:
            super().put(k, v)


def make_side(side, model, scene, n, max_steps, noise, autoreset=False, seed=5, skip_frames=1, **kw):
    _, spec, keep, low, high, A = scene_spec(scene, max_steps, noise, autoreset, seed, skip_frames)
    if side is GpuPrm and model.blob != load_scene(scene)[0].blob:
        # the GPU builds from a model handle: patch one with mjb_model_set_field
        m = load_scene(scene)[0]
        for k, v in L.parse_blob(model.blob).items():
            if v.dtype == np.float64 and not np.array_equal(v, m.fields[k]):
                m.set_field(k, v)
        assert m.blob == model.blob
        model = m
    reverse = kw.pop("reverse", False)
    return side(model, spec, keep, n, skip_frames, reverse, **kw), low, high, A


def no_damping(model):
    return not model.fields["dof_damping"].any()


def close(x, y):
    """the §3d tolerance: 1e-4 relative to max(1, |reference|)"""
    return bool((np.abs(x - y) / np.maximum(1.0, np.abs(y)) <= 1e-4).all())


# buffers not compared under the tolerance: the solver's warm start and iteration count (how it got there)
SOLVER_ONLY = ("warmstart", "niter")


def same(a, b, tag, names, approx=False):
    """bit for bit; with `approx` (models without damping) the float buffers within the §3d tolerance"""
    for k in names:
        if approx and k in SOLVER_ONLY:
            continue
        x, y = a.get(k), b.get(k)
        if approx and x.dtype == np.float32 and k != "params":
            assert close(x, y), (tag, k, np.abs(x - y).max())
        else:
            assert x.tobytes() == y.tobytes(), (tag, k)


def lower_free_bodies(side, model, drop=0.8):
    """move every free joint's body down by `drop`: the ants start on their legs, in contact with the floor"""
    f = model.fields
    q = side.get("qpos")
    for j in range(len(f["jnt_type"])):
        if int(f["jnt_type"][j]) == 0:
            q[:, int(f["jnt_qposadr"][j]) + 2] -= np.float32(drop)
    side.put("qpos", q)


def rand_act(side, rng, low, high, A):
    act = side.get("actions")
    act[:, :, :len(low)] = rng.uniform(low, high, (act.shape[0], A, len(low))).astype(np.float32)
    return act


# ---- 1. a neutral table changes nothing --------------------------------------------------------------------------------
def run_neutral(side, scene, n, noise, reverse=False, seed=5, steps=3):
    model = load_scene(scene)[0]
    kw = {} if side is GpuPrm else {"reverse": reverse}
    tab, low, high, A = make_side(side, model, scene, n, 50, noise, table=True, **kw)
    ref, _, _, _ = make_side(side, model, scene, n, 50, noise, **kw)
    approx = no_damping(model)
    names = ref.names
    rng = np.random.default_rng(seed)
    for s in (tab, ref):
        s.reset()
    same(tab, ref, "reset", names, approx)
    for t in range(steps):
        act = rand_act(ref, rng, low, high, A)
        for s in (tab, ref):
            s.put("actions", act)
            s.step()
        same(tab, ref, ("step", t), names, approx)
    for s in (tab, ref):
        s.forward()
    same(tab, ref, "forward", names, approx)
    if approx:   # the reset's draws are keyed by the rows: start both from the same ones
        for k in ref.names:
            tab.put(k, ref.get(k))
    for s in (tab, ref):
        s.reset((np.arange(n) % 3 == 1).astype(np.uint8))
    same(tab, ref, "masked reset", names, approx)
    assert tab.get("params").tobytes() == np.tile(model.nominal_params(), (n, 1)).tobytes()


@pytest.mark.parametrize("reverse", [False, True])
@pytest.mark.parametrize("noise", [0.0, 0.05])
@pytest.mark.parametrize("scene,n", [("2A", 4), ("S1", 8), ("C1", 4)])
def test_emulator_neutral_table_is_bit_identical(scene, n, noise, reverse):
    run_neutral(EmuPrm, scene, n, noise, reverse)


# ---- 2. an env with its own row is the env of a model compiled with that row -------------------------------------------
def random_rows(model, n, rng, spread=0.3):
    nom = model.nominal_params()
    return (nom[None, :] * rng.uniform(1 - spread, 1 + spread, (n, nom.size))).astype(np.float32)


def run_rows(side, scene, n, noise, reverse=False, seed=5, steps=4, distinct=None):
    """every env (or the envs in `distinct`, the others nominal) gets its own row; env e must equal env e of a batch of
    the blob patched to that row, over `steps` steps with contacts"""
    model = load_scene(scene)[0]
    kw = {} if side is GpuPrm else {"reverse": reverse}
    rng = np.random.default_rng(seed)
    rows = np.tile(model.nominal_params(), (n, 1)).astype(np.float32)
    distinct = np.arange(n) if distinct is None else np.asarray(distinct)
    rows[distinct] = random_rows(model, len(distinct), rng)
    tab, low, high, A = make_side(side, model, scene, n, 10 ** 6, noise, table=True, **kw)
    tab.put("params", rows)
    acts = [rand_act(tab, rng, low, high, A) for _ in range(steps)]
    tab.reset()
    if scene != "S1":
        lower_free_bodies(tab, model)
    out = [{k: tab.get(k) for k in tab.names}]
    for a in acts:
        tab.put("actions", a)
        tab.step()
        out.append({k: tab.get(k) for k in tab.names})
    assert np.max([o["ncon"][distinct] for o in out], axis=0).min() > 0   # every env with its own row touched something
    approx = no_damping(model)
    groups = {}
    for e in distinct:
        groups.setdefault(rows[e].tobytes(), []).append(e)
    if len(distinct) < n:
        groups.setdefault(model.nominal_params().tobytes(), []).extend(sorted(set(range(n)) - set(distinct.tolist())))
    for key, envs in groups.items():
        row = np.frombuffer(key, np.float32)
        ref, _, _, _ = make_side(side, _BlobModel(model, patched_blob(model, row)), scene, n, 10 ** 6, noise, **kw)
        ref.reset()
        if scene != "S1":
            lower_free_bodies(ref, model)
        snaps = [{k: ref.get(k) for k in ref.names}]
        for a in acts:
            ref.put("actions", a)
            ref.step()
            snaps.append({k: ref.get(k) for k in ref.names})
        for t, (o, r) in enumerate(zip(out, snaps)):
            for k in r:
                if approx and k in SOLVER_ONLY:
                    continue
                x, y = o[k][envs], r[k][envs]
                if approx and x.dtype == np.float32:
                    assert close(x, y), (t, k, envs)
                else:
                    assert x.tobytes() == y.tobytes(), (t, k, envs)
    assert out[-1]["params"].tobytes() == rows.tobytes()   # rows persist without randomisation


@pytest.mark.parametrize("reverse", [False, True])
@pytest.mark.parametrize("noise", [0.0, 0.05])
@pytest.mark.parametrize("scene,n", [("2A", 2), ("S1", 4), ("C1", 4)])
def test_emulator_rows_equal_patched_models(scene, n, noise, reverse):
    run_rows(EmuPrm, scene, n, noise, reverse)


# ---- 3. randomising resets = numpy draws written as rows + resets without randomisation ----------------------------------
RANGES = [(0.7, 1.3), (0.5, 1.5), (0.8, 1.2), (0.0, 2.0)]


def run_random(side, scene, n, noise, steps, max_steps, reverse=False, seed=5):
    model = load_scene(scene)[0]
    kw = {} if side is GpuPrm else {"reverse": reverse}
    rnd, low, high, A = make_side(side, model, scene, n, max_steps, noise, autoreset=True, seed=seed, ranges=RANGES, **kw)
    ref, _, _, _ = make_side(side, model, scene, n, max_steps, noise, seed=seed, table=True, **kw)
    names = ref.names
    e = np.arange(n)
    # full reset: keys from the rows before it
    ep = reset_key_np(ref.get("timestep"), ref.get("qpos")[:, 0], ref.get("qvel")[:, 0])
    ref.put("params", drawn_rows(model, ref.get("params"), seed, e, ep, RANGES))
    for s in (rnd, ref):
        s.reset()
    same(rnd, ref, "randomising reset", names)
    assert rnd.get("params").tobytes() != np.tile(model.nominal_params(), (n, 1)).tobytes()
    # masked reset
    rng = np.random.default_rng(seed)
    for s in (rnd, ref):
        s.put("actions", rand_act(ref, rng, low, high, A)) if s is rnd else None
    act = rnd.get("actions")
    ref.put("actions", act)
    for s in (rnd, ref):
        s.put("timestep", ((e // 4 * 7 + e % 4) % max_steps).astype(np.int32))
    mask = (e % 3 == 1).astype(np.uint8)
    m = np.nonzero(mask)[0]
    ep = reset_key_np(ref.get("timestep")[m], ref.get("qpos")[m, 0], ref.get("qvel")[m, 0])
    p = ref.get("params")
    p[m] = drawn_rows(model, p[m], seed, m, ep, RANGES)
    ref.put("params", p)
    for s in (rnd, ref):
        s.reset(mask)
    same(rnd, ref, "randomising masked reset", names)
    # reset from the caller's rows (mjb_reset_rows): the keys read those rows
    mask = (e % 3 == 2).astype(np.uint8)
    m = np.nonzero(mask)[0]
    rows_q, rows_v = ref.get("qpos"), ref.get("qvel")
    rows_q, rows_v = rows_q[np.roll(e, 1)], rows_v[np.roll(e, 1)]   # every env gets another env's state
    for s in (rnd, ref):
        q, v = s.get("qpos"), s.get("qvel")
        q[m], v[m] = rows_q[m], rows_v[m]
        s.put("qpos", q)
        s.put("qvel", v)
    ep = reset_key_np(ref.get("timestep")[m], rows_q[m, 0], rows_v[m, 0])
    p = ref.get("params")
    p[m] = drawn_rows(model, p[m], seed, m, ep, RANGES)
    ref.put("params", p)
    for s in (rnd, ref):
        s.reset_rows(mask)
    same(rnd, ref, "randomising reset from rows", names)
    for s in (rnd, ref):
        s.put("timestep", ((e // 4 * 7 + e % 4) % max_steps).astype(np.int32))
    # auto-resets: plain step, draw the finished envs' rows and actions, masked reset, flags put back
    ended = 0
    for t in range(steps):
        act = rand_act(ref, rng, low, high, A)
        rnd.put("actions", act)
        ref.put("actions", act)
        rnd.step()
        ref.step()
        saved = {k: ref.get(k) for k in ("reward", "term", "trunc")}
        fin = (saved["term"][:, A] | saved["trunc"][:, A]).astype(bool)
        if fin.any():
            env = np.nonzero(fin)[0]
            ep = reset_key_np(ref.get("timestep")[env], ref.get("qpos")[env, 0], ref.get("qvel")[env, 0])
            p = ref.get("params")
            p[env] = drawn_rows(model, p[env], seed, env, ep, RANGES)
            ref.put("params", p)
            drawn = act.copy()
            for a in range(A):
                for d in range(len(low)):
                    drawn[env, a, d] = reset_action_np(seed, env, a, d, ep, low[d], high[d])
            ref.put("actions", drawn)
            ref.reset(fin.astype(np.uint8))
            ref.put("actions", act)
            for k, v in saved.items():
                ref.put(k, v)
            ended += len(env)
        same(rnd, ref, ("auto-reset step", t), names)
    return ended


@pytest.mark.parametrize("reverse", [False, True])
@pytest.mark.parametrize("noise", [0.0, 0.05])
@pytest.mark.parametrize("scene,n,steps,max_steps", [("2A", 4, 5, 4), ("S1", 8, 5, 3), ("C1", 4, 5, 3)])
def test_emulator_randomising_resets_equal_drawn_rows(scene, n, steps, max_steps, noise, reverse):
    assert run_random(EmuPrm, scene, n, noise, steps, max_steps, reverse) >= n // 2


# ---- 4. the exported draw, the layout, the model edit, the refusals ----------------------------------------------------
def test_param_scale_export_matches_numpy_restatement():
    lib = L.load()
    rng = np.random.default_rng(4)
    for _ in range(300):
        seed, env, fam, idx, ep = int(rng.integers(0, 2 ** 63)), int(rng.integers(0, 1 << 20)), int(rng.integers(0, 4)), \
            int(rng.integers(0, 4096)), int(rng.integers(0, 2 ** 32))
        lo = np.float32(rng.uniform(0.01, 1))
        hi = np.float32(lo + rng.uniform(0, 2))
        want = np.asarray(param_scale_np(seed, env, fam, idx, ep, lo, hi), np.float32)
        got = np.float32(lib.mjb_param_scale(seed, env, fam, idx, ep, lo, hi))
        assert got.view(np.uint32) == want.view(np.uint32)
        assert lo <= got <= hi
    assert lib.mjb_param_scale(1, 2, 3, 4, 5, 1.0, 1.0) == 1.0


def test_param_layout_and_nominal_row():
    model = load_scene("2A")[0]
    lay, f = model.param_layout(), model.fields
    nb, ng = model.nbody, model.ngeom
    assert (lay.body_mass, lay.body_inertia, lay.geom_friction, lay.actuator_gear, lay.dof_damping, lay.n_params) == \
        (0, nb, 4 * nb, 4 * nb + ng, 4 * nb + ng + model.nu, 4 * nb + ng + model.nu + model.nv)
    row = model.nominal_params()
    assert row.dtype == np.float32 and row.size == lay.n_params
    assert (row[lay.geom_friction:lay.geom_friction + ng] == f["geom_friction"][0::3].astype(np.float32)).all()
    assert (row[lay.dof_damping:] == f["dof_damping"].astype(np.float32)).all()


def test_model_set_field():
    model = load_scene("2A")[0]
    blob = model.blob
    for k in ("body_mass", "body_inertia", "geom_friction", "actuator_gear", "dof_damping", "pair_friction"):
        model.set_field(k, model.fields[k])
    assert model.blob == blob   # unchanged values: byte-identical blob
    m2 = model.fields["body_mass"].copy()
    m2[2] *= 2
    model.set_field("body_mass", m2)
    assert model.fields["body_mass"][2] == m2[2]
    assert (model.fields["body_invweight0"] == L.parse_blob(blob)["body_invweight0"]).all()   # nothing derived recomputed
    # geom friction reaches the contacts: the pairs' mixed friction is the elementwise max of the geoms'
    f = model.fields
    gf = f["geom_friction"].copy()
    gf[0::3] *= np.linspace(0.5, 2.0, model.ngeom)
    model.set_field("geom_friction", gf)
    g = model.fields["geom_friction"].reshape(-1, 3)
    want = np.maximum(g[f["pair_geom1"]], g[f["pair_geom2"]]).reshape(-1)
    assert f["pair_geom1"].size and np.array_equal(model.fields["pair_friction"], want)
    for name, vals in (("no_such_field", [1.0]), ("body_parentid", model.fields["body_parentid"]), ("body_mass", m2[:-1])):
        with pytest.raises(Exception):
            model.set_field(name, vals)


def test_refusals():
    lib = emu_params_lib()
    model = load_scene("2A")[0]
    _, spec, keep, _, _, _ = scene_spec("2A", 50, 0.0, False)
    table = np.zeros((1, model.param_layout().n_params), np.float32)

    def err(**kw):
        s = L.EnvSpec.from_buffer_copy(spec)
        s.params = kw.get("params", table.ctypes.data)
        s.skip_frames = kw.get("skip", 1)
        if "ranges" in kw:
            s.flags |= L.SPEC_RANDOMIZE
            for f, (lo, hi) in enumerate(kw["ranges"]):
                s.param_lo[f], s.param_hi[f] = lo, hi
        return lib.emu_param_spec_error(ctypes.byref(s)).decode()
    ok = [(1.0, 1.0)] * 4
    assert err() == "" and err(ranges=ok) == "" and err(ranges=[(0.5, 2.0), (0.0, 1.0), (0.0, 0.0), (0.0, 3.0)]) == ""
    assert "needs spec.params" in err(params=None, ranges=ok)
    assert "skip_frames" in err(skip=0)
    assert "finite" in err(ranges=[(1.0, float("inf"))] + ok[1:])
    assert "finite" in err(ranges=ok[:1] + [(float("nan"), 1.0)] + ok[2:])
    assert "<=" in err(ranges=ok[:2] + [(1.5, 1.0)] + ok[3:])
    assert ">= 0" in err(ranges=ok[:3] + [(-0.1, 1.0)])
    assert "> 0 for body mass" in err(ranges=[(0.0, 1.0)] + ok[1:])


def test_config_validation():
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import parse_param_ranges
    assert parse_param_ranges(None) is None
    assert parse_param_ranges({}) == [(1.0, 1.0)] * 4
    assert parse_param_ranges({"geom_friction": [0.5, 1.5]}) == [(1.0, 1.0), (0.5, 1.5), (1.0, 1.0), (1.0, 1.0)]
    for bad in ({"body_masses": [1, 1]}, [0.5, 1.5], {"body_mass": [0.0, 1.0]}, {"dof_damping": [-1, 1]},
                {"actuator_gear": [2, 1]}, {"geom_friction": [1, float("inf")]}, {"geom_friction": 1.0}, {"geom_friction": [1]}):
        with pytest.raises(Exception):
            parse_param_ranges(bad)


# ---- GPU ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("scene", ["2A", "C1", "S1"])
def test_gpu_neutral_table_is_bit_identical(scene):
    run_neutral(GpuPrm, scene, 4096, 0.05)


@pytest.mark.gpu
@pytest.mark.parametrize("scene", ["2A", "C1", "S1"])
def test_gpu_rows_equal_patched_models(scene):
    rng = np.random.default_rng(1)
    run_rows(GpuPrm, scene, 4096, 0.0, distinct=np.sort(rng.choice(4096, 6, replace=False)))


@pytest.mark.gpu
@pytest.mark.parametrize("scene", ["2A", "C1", "S1"])
def test_gpu_randomising_resets_equal_drawn_rows(scene):
    assert run_random(GpuPrm, scene, 4096, 0.05, 6, 4) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("scene", ["2A", "C1"])
def test_gpu_matches_fp64_oracle_on_patched_model(scene):
    """one step of envs with their own rows against the fp64 oracle run on the blob patched to that row (§3d tolerance)"""
    import torch
    from oracle import OracleSim
    from test_gpu_parity import RTOL, rel_err
    model, tables, agents, fj = load_scene(scene)
    n, nq, nv, nu = 256, model.nq, model.nv, model.nu
    rng = np.random.default_rng(9)
    envs = [3, 77, 200]
    rows = random_rows(model, len(envs), rng)
    gpu, low, high, A = make_side(GpuPrm, model, scene, n, 10 ** 6, 0.0, table=True)
    p = gpu.get("params")
    p[envs] = rows
    gpu.put("params", p)
    gpu.reset()
    for _ in range(6):
        gpu.put("actions", rand_act(gpu, rng, low, high, A))
        gpu.b.physics(1)
    pre = {k: gpu.get(k).astype(np.float64) for k in ("qpos", "qvel", "warmstart", "ctrl")}
    act = rand_act(gpu, rng, low, high, A)
    gpu.put("actions", act)
    gpu.b.physics(1)
    q, v, ncon, cg = gpu.get("qpos"), gpu.get("qvel"), gpu.get("ncon"), gpu.get("contact_geom")
    n_phys = len(tables.act_space[agents[0]]["low"])
    for e, row in zip(envs, rows):
        sim = OracleSim(patched_blob(model, row))
        sim.qpos[:] = pre["qpos"][e, :nq]; sim.qvel[:] = pre["qvel"][e, :nv]; sim.qacc_warmstart[:] = pre["warmstart"][e, :nv]
        if nu:
            sim.ctrl[:] = pre["ctrl"][e, :nu]
        for a, agent in enumerate(agents):
            idx = tables.agents_action_index[agent]
            if fj:
                sim.qvel[idx] = act[e, a, :n_phys]
            else:
                sim.ctrl[idx] = act[e, a, :n_phys]
        sim.step()
        assert rel_err(q[e, :nq], sim.qpos) < RTOL and rel_err(v[e, :nv], sim.qvel) < RTOL, (scene, e)
        assert sorted((int(x), int(y)) for x, y in cg[e, :ncon[e]]) == sorted(sim.contact_pairs()), (scene, e)


@pytest.mark.gpu
def test_gpu_python_api():
    import torch
    from mujoco_rl_environment_wrapper_b200 import plugins as P
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL
    lv = LEVELS
    base = {"xmlPath": os.path.join(lv, "two_ants.xml"), "infoJson": os.path.join(lv, "info_2A.json"), "agents": ["sender", "receiver"],
            "environmentDynamics": [P.Language], "rewardFunctions": [P.tag_distance_reward], "doneFunctions": [P.distance_done]}
    # N > 1: views, writes take effect at the next step
    env = MuJoCoRL({**base, "num_envs": 64, "perEnvParams": True, "seed": 3})
    nb, ng = env.model.nbody, env.model.ngeom
    assert env.params["body_mass"].shape == (64, nb) and env.params["body_inertia"].shape == (64, nb, 3)
    assert env.params["geom_friction"].shape == (64, ng) and env.params["actuator_gear"].shape == (64, env.model.nu)
    assert env.params["dof_damping"].shape == (64, env.model.nv)
    twin = MuJoCoRL({**base, "num_envs": 64, "seed": 3})
    env.reset()
    twin.reset()
    acts = env.sample_actions()
    env.params["actuator_gear"][5] *= 3.0
    env.step(acts)
    twin.step(acts)
    qa, qb = env.batch.qpos, twin.batch.qpos
    assert not torch.equal(qa[5], qb[5]) and torch.equal(torch.cat([qa[:5], qa[6:]]), torch.cat([qb[:5], qb[6:]]))
    assert float(env.model.fields["actuator_gear"][0]) == float(twin.model.fields["actuator_gear"][0])   # env.model stays nominal
    # N = 1: squeezed views
    one = MuJoCoRL({**base, "num_envs": 1, "perEnvParams": True})
    assert one.params["body_mass"].shape == (nb,) and one.params["body_inertia"].shape == (nb, 3)
    one.params["body_mass"][2] = 10.0
    assert float(one.batch.params[0, 2]) == 10.0
    # randomizeParams with autoReset and startStates
    f = env.model.fields
    pool = {"qpos": np.tile(f["qpos0"][:env.model.nq], (3, 1))}
    rnd = MuJoCoRL({**base, "num_envs": 256, "autoReset": True, "startStates": pool, "maxSteps": 3,
                    "randomizeParams": {"body_mass": [0.8, 1.2], "geom_friction": [0.5, 1.5]}})
    rnd.reset()
    m0 = rnd.params["body_mass"].clone()
    assert not torch.equal(m0[0], m0[1])
    g = rnd.params["actuator_gear"]
    assert torch.equal(g, g[:1].expand_as(g))   # (1, 1): nominal
    for _ in range(4):
        rnd.step(rnd.sample_actions())
    assert not torch.equal(rnd.params["body_mass"], m0)   # the auto-resets drew new rows
    assert torch.isfinite(rnd.batch.qpos).all()
    with pytest.raises(Exception):
        MuJoCoRL({**base, "num_envs": 4, "randomizeParams": {"body_mass": [0.0, 1.0]}})


@pytest.mark.gpu
def test_gpu_level_variants_share_one_table():
    import torch
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL
    lv = LEVELS
    env = MuJoCoRL({"xmlPath": [os.path.join(lv, "two_ants.xml"), os.path.join(lv, "two_ants_cams.xml")],
                    "infoJson": os.path.join(lv, "info_2A.json"), "agents": ["sender", "receiver"], "num_envs": 64,
                    "randomizeParams": {"body_mass": [0.9, 1.1]}})
    b0, b1 = env._levels[0]["batch"], env._levels[1]["batch"]
    assert b0.params.data_ptr() == b1.params.data_ptr()
    env.reset()
    env.step(env.sample_actions())
    assert torch.isfinite(env.batch.qpos).all()


@pytest.mark.gpu
def test_gpu_level_variants_with_different_physics(tmp_path):
    """two levels whose joints differ in damping and whose actuators differ in gear: without randomisation every env's row
    holds its own level's values (written when the env moves to a level), so the batch equals the single-level batches
    of each level, bit for bit; rows the caller wrote persist while the env stays on its level"""
    import torch
    from mujoco_rl_environment_wrapper_b200 import plugins as P
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL
    a = open(os.path.join(LEVELS, "two_ants.xml")).read()
    b = a.replace('damping="1"', 'damping="2.5"', 1).replace('gear="150"', 'gear="120"', 4)
    assert b.count('gear="120"') == 4 and 'damping="2.5"' in b
    xa, xb = str(tmp_path / "A.xml"), str(tmp_path / "B.xml")
    open(xa, "w").write(a)
    open(xb, "w").write(b)
    ja = os.path.join(LEVELS, "info_2A.json")
    common = dict(agents=["sender", "receiver"], environmentDynamics=[P.Language], rewardFunctions=[P.tag_distance_reward],
                  doneFunctions=[P.distance_done], infoJson=ja, num_envs=96, seed=7)
    multi = MuJoCoRL(dict(common, xmlPath=[xa, xb], perEnvParams=True))
    singles = [MuJoCoRL(dict(common, xmlPath=xa)), MuJoCoRL(dict(common, xmlPath=xb))]
    nom = [torch.from_numpy(lv["model"].nominal_params()).cuda() for lv in multi._levels]
    assert not torch.equal(nom[0], nom[1])
    table = multi.batch.params

    def rows_follow_levels():
        lid = multi.level_id.long()
        return torch.equal(table, torch.where((lid == 0)[:, None], nom[0][None, :], nom[1][None, :]))
    envs = [multi] + singles
    for e in envs:
        e.reset()
    lid = multi.level_id.cpu().numpy()
    assert set(lid.tolist()) == {0, 1} and rows_follow_levels()
    for t in range(20):
        acts = [e.sample_actions() for e in envs]
        for e, act in zip(envs, acts):
            e.step(act)
        for name in ("qpos", "qvel", "obs", "reward", "term", "trunc"):
            got = getattr(multi.batch, name).cpu().numpy()
            want = np.where(lid.reshape((-1,) + (1,) * (got.ndim - 1)) == 0, getattr(singles[0].batch, name).cpu().numpy(),
                            getattr(singles[1].batch, name).cpu().numpy())
            assert got.tobytes() == np.ascontiguousarray(want).tobytes(), (t, name)
    assert not torch.equal(singles[0].batch.qpos, singles[1].batch.qpos)   # the levels' physics differ
    # a masked reset moves some envs to the other level: those get its values, the others keep what the caller wrote
    table[:, 0] = 123.0   # body 0 (the world): an entry the kernel ignores, used here as a marker
    mask = torch.zeros(96, dtype=torch.bool)
    mask[::2] = True
    multi.reset(mask=mask)
    lid2 = multi.level_id.cpu().numpy()
    moved = torch.from_numpy(lid2 != lid).cuda()
    assert bool(moved.any()) and bool((~moved & mask.cuda()).any())
    assert torch.equal(table[~moved, 0], torch.full_like(table[~moved, 0], 123.0))
    expect = torch.where(torch.from_numpy(lid2 == 0).cuda()[:, None], nom[0][None, :], nom[1][None, :])
    assert torch.equal(table[moved], expect[moved])


@pytest.mark.gpu
def test_gpu_65536_env_randomised_rollout_stays_finite():
    import torch
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL
    from mujoco_rl_environment_wrapper_b200 import plugins as P
    r = [0.7, 1.3]
    env = MuJoCoRL({"xmlPath": os.path.join(LEVELS, "two_ants.xml"), "infoJson": os.path.join(LEVELS, "info_2A.json"),
                    "agents": ["sender", "receiver"], "environmentDynamics": [P.Language], "rewardFunctions": [P.tag_distance_reward],
                    "doneFunctions": [P.distance_done], "num_envs": 65536, "autoReset": True, "maxSteps": 20,
                    "randomizeParams": {k: r for k in L.PARAM_FAMILIES}})
    env.reset()
    m0 = env.params["body_mass"].clone()
    for _ in range(50):
        env.step(env.sample_actions())
    assert not torch.equal(env.params["body_mass"], m0)
    b = env.batch
    assert torch.isfinite(b.qpos).all() and torch.isfinite(b.qvel).all() and torch.isfinite(b.obs).all()
    assert int(b.nreset.sum()) == 0
