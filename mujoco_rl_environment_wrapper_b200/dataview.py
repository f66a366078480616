"""`env.data` / `env.model` views for plugin code written against the reference's `mujoco` objects.

The reference hands plugins the environment itself, and plugins reach through it into `MjData` / `MjModel`
(benchmarking/fps_gym/fps_custom_env.py:20-23: `env.model.opt.timestep`, `env.data.ctrl`, `env.data.cfrc_ext`;
Testing/Pick_Up_Dynamic.py:40: `data.body(name).xipos`; mujoco_parent.py:404-425,441-443,463-475).  Here the state
lives in the batch's CUDA tensors; these classes expose it under the same attribute names:

  * `num_envs == 1`: numpy float64 arrays / Python scalars with the reference's shapes (copies: read-only views of
    the device state), so code written for the reference runs unmodified;
  * `num_envs  > 1`: CUDA tensors with a leading env dimension (views, no copy).

Positions (`xipos`, `xpos`) exist for the exported objects: the agents, every object tagged "target" in the info
JSON, whatever `config_dict["exportPositions"]` lists, and every STATIC object (a constant).  They come from the last
forward pass of the step, exactly what `data.xipos` holds after `mj_step`.
"""
import types

import numpy as np
import torch

from . import _lib as L


def quat_mul(a, b):
    return np.array([a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3], a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2],
                     a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1], a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0]])


def quat_rot(q, v):
    w, u = q[0], np.asarray(q[1:])
    t = 2.0 * np.cross(u, v)
    return v + w * t + np.cross(u, t)


def static_pose(fields, objtype, oid):
    """world pose (pos, quat, ipos) of a body / geom that cannot move (no joint between it and the world), else None"""
    body = oid if objtype == L.OBJ_BODY else int(fields["geom_bodyid"][oid])
    if int(fields["body_weldid"][body]) != 0:
        return None
    chain = []
    b = body
    while b > 0:
        chain.append(b)
        b = int(fields["body_parentid"][b])
    pos, quat = np.zeros(3), np.array([1.0, 0, 0, 0])
    for b in reversed(chain):
        pos = pos + quat_rot(quat, fields["body_pos"][3 * b:3 * b + 3])
        quat = quat_mul(quat, fields["body_quat"][4 * b:4 * b + 4])
    if objtype == L.OBJ_BODY:
        return pos + quat_rot(quat, fields["body_ipos"][3 * body:3 * body + 3]), quat
    return pos + quat_rot(quat, fields["geom_pos"][3 * oid:3 * oid + 3]), quat_mul(quat, fields["geom_quat"][4 * oid:4 * oid + 4])


def quat_to_euler_zyx_deg(q):
    """scipy's Rotation.as_euler("zyx", degrees=True) of the rotation `q` (w, x, y, z): intrinsic... the reference's
    helper.mat2euler_scipy (MuJoCo_Gym/helper.py:6-18).  Batched over leading dimensions (torch or numpy)."""
    is_t = torch.is_tensor(q)
    xp = torch if is_t else np
    w, x, y, z = q[..., 0], q[..., 1], q[..., 2], q[..., 3]
    # extrinsic z, then y, then x  ==  R = Rx(c) Ry(b) Rz(a);  R[0][2] = sin(b)
    r02 = 2 * (x * z + w * y)
    r01, r00 = 2 * (x * y - w * z), 1 - 2 * (y * y + z * z)
    r12, r22 = 2 * (y * z - w * x), 1 - 2 * (x * x + y * y)
    b = xp.arcsin(xp.clip(r02, -1.0, 1.0)) if not is_t else torch.asin(torch.clamp(r02, -1.0, 1.0))
    a = (xp.arctan2(-r01, r00) if not is_t else torch.atan2(-r01, r00))
    c = (xp.arctan2(-r12, r22) if not is_t else torch.atan2(-r12, r22))
    out = xp.stack([a, b, c], -1) if is_t else np.stack([a, b, c], -1)
    return out * (180.0 / np.pi)


class _Named(types.SimpleNamespace):
    pass


class ModelView:
    """`env.model`: the compiled model (L.Model) plus the `MjModel` attribute names plugins use."""

    def __init__(self, model):
        self._m = model
        self.opt = types.SimpleNamespace(timestep=float(model.timestep), gravity=np.array(model.fields["opt_gravity"]))
        for k in ("nq", "nv", "nu", "nbody", "njnt", "ngeom", "nsite", "nsensor", "nsensordata"):
            setattr(self, k, getattr(model, k))

    def __getattr__(self, k):   # everything else (name2id, fields, blob, dims ...) is the compiled model's
        return getattr(self._m, k)

    def _id(self, objtype, name, what):
        if isinstance(name, (int, np.integer)):
            return int(name)
        i = self._m.name2id(objtype, name)
        if i < 0:
            raise KeyError(f"Invalid name '{name}' for {what}")
        return i

    def body(self, name):
        i = self._id(L.OBJ_BODY, name, "body")
        f = self._m.fields
        return _Named(id=i, name=self._m.id2name(L.OBJ_BODY, i), mass=np.array([f["body_mass"][i]]), pos=f["body_pos"][3 * i:3 * i + 3].copy(),
                      parentid=int(f["body_parentid"][i]))

    def geom(self, name):
        i = self._id(L.OBJ_GEOM, name, "geom")
        f = self._m.fields
        return _Named(id=i, name=self._m.id2name(L.OBJ_GEOM, i), rgba=f["geom_rgba"][4 * i:4 * i + 4].astype(np.float32), type=np.array([f["geom_type"][i]]),
                      size=f["geom_size"][3 * i:3 * i + 3].copy(), bodyid=int(f["geom_bodyid"][i]))

    def joint(self, name):
        i = self._id(L.OBJ_JOINT, name, "joint")
        f = self._m.fields
        return _Named(id=i, name=self._m.id2name(L.OBJ_JOINT, i), dofadr=np.array([f["jnt_dofadr"][i]]), qposadr=np.array([f["jnt_qposadr"][i]]),
                      type=np.array([f["jnt_type"][i]]))

    def camera(self, name):
        return _Named(id=self._id(L.OBJ_CAMERA, name, "camera"), name=name)

    def sensor(self, name):
        i = self._id(L.OBJ_SENSOR, name, "sensor")
        f = self._m.fields
        return _Named(id=i, name=self._m.id2name(L.OBJ_SENSOR, i), type=np.array([f["sensor_type"][i]]),
                      adr=np.array([f["sensor_adr"][i]]), dim=np.array([f["sensor_dim"][i]]),
                      objtype=np.array([f["sensor_objtype"][i]]), objid=np.array([f["sensor_objid"][i]]),
                      cutoff=np.array([f["sensor_cutoff"][i]]))


class _Contact:
    def __init__(self, g1, g2, dist):
        self.geom1, self.geom2, self.dist = g1, g2, dist


class DataView:
    """`env.data`: `MjData` attribute names over the batch tensors (see the module docstring for shapes)."""

    def __init__(self, env):
        self._env = env

    def _out(self, t):
        if self._env.num_envs > 1:
            return t
        return t[0].detach().cpu().numpy().astype(np.float64)

    @property
    def qpos(self):
        return self._out(self._env._batch.qpos[:, :self._env.model.nq])

    @property
    def qvel(self):
        return self._out(self._env._batch.qvel[:, :self._env.model.nv])

    @property
    def ctrl(self):
        return self._out(self._env._batch.ctrl[:, :self._env.model.nu])

    @property
    def sensordata(self):
        return self._out(self._env._batch.sensordata[:, :self._env.model.nsensordata])

    @property
    def qacc_warmstart(self):
        return self._out(self._env._batch.warmstart[:, :self._env.model.nv])

    @property
    def cfrc_ext(self):
        """MuJoCo fills cfrc_ext only when the model has force / torque / accelerometer sensors (mj_rnePostConstraint);
        for every other model it is identically zero, which is what this returns.  Models with such sensors raise."""
        env = self._env
        if any(int(t) == 1 for t in env.model.fields["sensor_type"]):
            raise NotImplementedError("data.cfrc_ext: the model has accelerometer sensors, for which MuJoCo computes body contact wrenches; "
                                      "this implementation does not export them")
        n = env.model.nbody
        return np.zeros((n, 6)) if env.num_envs == 1 else torch.zeros((env.num_envs, n, 6), device=env.device)

    @property
    def time(self):
        t = self._env._batch.timestep.to(torch.float64) * float(self._env.model.timestep) * max(1, int(self._env.skip_frames))
        return t if self._env.num_envs > 1 else float(t[0])

    @property
    def ncon(self):
        n = self._env._batch.ncon
        return n if self._env.num_envs > 1 else int(n[0])

    @property
    def contact(self):
        """num_envs == 1: list of contacts with `.geom1 / .geom2 / .dist` (mujoco_parent.py:472-475);
        otherwise the raw tensors (geom pairs [N, maxcon, 2], valid where index < ncon)"""
        b = self._env._batch
        if self._env.num_envs > 1:
            return b.contact_geom
        n = int(b.ncon[0])
        cg, cd = b.contact_geom[0, :n].cpu().numpy(), b.contact_dist[0, :n].cpu().numpy()
        return [_Contact(int(cg[i, 0]), int(cg[i, 1]), float(cd[i])) for i in range(n)]

    def body(self, name):
        env = self._env
        i = env.model._id(L.OBJ_BODY, name, "body")
        nm = env.model.id2name(L.OBJ_BODY, i)
        return _LazyObject(env, nm, L.OBJ_BODY, i)

    def geom(self, name):
        env = self._env
        i = env.model._id(L.OBJ_GEOM, name, "geom")
        nm = env.model.id2name(L.OBJ_GEOM, i)
        return _LazyObject(env, nm, L.OBJ_GEOM, i)

    def sensor(self, name):
        """`data.sensor(n)`: id, name and `.data`, the sensor's slice of sensordata (numpy for one env, a [N, dim] view)"""
        env = self._env
        i = env.model._id(L.OBJ_SENSOR, name, "sensor")
        f = env.model.fields
        adr, dim = int(f["sensor_adr"][i]), int(f["sensor_dim"][i])
        return _Named(id=i, name=env.model.id2name(L.OBJ_SENSOR, i), data=self._out(env._batch.sensordata[:, adr:adr + dim]))


class _LazyObject:
    """`data.body(n)` / `data.geom(n)`: id, name, xipos | xpos, xmat (computed on access)"""

    def __init__(self, env, name, objtype, oid):
        self._env, self.name, self._ot, self.id = env, name, objtype, oid

    def _pos(self):
        return self._env._out(self._env._position(self.name))

    @property
    def xipos(self):
        if self._ot != L.OBJ_BODY:
            raise AttributeError("xipos")
        return self._pos()

    @property
    def xpos(self):
        if self._ot == L.OBJ_GEOM:
            return self._pos()
        raise NotImplementedError("data.body(n).xpos (frame origin) is not exported; xipos (centre of mass) is")

    @property
    def xmat(self):
        q = self._env._orientation_quat(self.name)
        w, x, y, z = q[..., 0], q[..., 1], q[..., 2], q[..., 3]
        rows = [1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y), 2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x),
                2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]
        m = torch.stack(rows, -1) if torch.is_tensor(q) else np.stack(rows, -1)
        return self._env._out(m) if torch.is_tensor(m) else m
