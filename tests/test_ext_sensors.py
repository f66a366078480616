"""Frame, velocity and joint sensors (gyro, velocimeter, jointpos / jointvel, framepos / framequat / framelinvel /
frameangvel, frame axes of bodies and geoms): compiler against an independent derivation, refusals, closed forms of the
fp64 reference, the device step code (SIMT emulator on the CPU, the CUDA batch on the GPU) against it, the observation
tables and the Python API.

The reference (`SensorRef`, below) restates the new sensors in fp64 from the CPU oracle's matrix kinematics (body, geom
and site frames after `orc_forward`) and a world-frame point Jacobian built from them, without the kernel's spatial
recursion.  The oracle itself only evaluates the sensors it has always known (touch, accelerometer, rangefinder, frame
axes of sites): it runs on the same level with every other sensor removed, which changes no physics, and those sensors
are compared from its `sensordata`.  Tolerance as DESIGN §3d: |x - x_ref| <= 1e-4 * max(1, |x_ref|), acceleration-stage
sensors 2e-3 (as test_gpu_parity.py); framequat is compared through quat2mat with the reference's rotation matrix.
The fixtures live in tests/sensor_levels/: tests/levels/ holds the scenes the full-blob derivation of
oracle/model_ref.py knows."""
import math
import os
import re
import xml.etree.ElementTree as ET

import numpy as np
import pytest

import emu_harness as E
from common import LEVELS, make_spec
from mujoco_rl_environment_wrapper_b200 import _lib as L
from mujoco_rl_environment_wrapper_b200.tables import Tables
from oracle import OracleSim
from oracle.model_ref import RefModel, quat2mat

SENSOR_LEVELS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "sensor_levels")
FIELDS = ("sensor_type", "sensor_objtype", "sensor_objid", "sensor_adr", "sensor_dim", "sensor_datatype", "sensor_cutoff")
T = L.SENSOR_TYPE
AXES = ("framexaxis", "frameyaxis", "framezaxis")
# name: (xml, agents, free_joint)
LEVELS_IMU = {"box_imu": ("box_imu.xml", ["receiver"], True), "two_ants_imu": ("two_ants_imu.xml", ["sender", "receiver"], False),
              "ant_rk4_imu": ("ant_rk4_imu.xml", ["torso"], False)}
RTOL, ACC_TOL = 1e-4, 2e-3


def level_text(name):
    return open(os.path.join(SENSOR_LEVELS, LEVELS_IMU[name][0])).read()


def load(name):
    _, agents, fj = LEVELS_IMU[name]
    text = level_text(name)
    model = L.Model(text)
    return model, Tables(text, model, agents, fj), agents, fj


def rel_err(x, ref):
    x, ref = np.asarray(x, float), np.asarray(ref, float)
    return float((np.abs(x - ref) / np.maximum(1.0, np.abs(ref))).max()) if ref.size else 0.0


def _legacy(el):
    """a sensor the CPU oracle evaluates itself"""
    return el.tag in ("touch", "accelerometer", "rangefinder") or (el.tag in AXES and el.get("objtype") == "site")


class SensorRef:
    """Independent derivation of the seven sensor fields from the XML (ElementTree + the object lists of
    oracle.model_ref.RefModel), and the fp64 values of the new sensors from the oracle's kinematics."""
    TAGS = {"touch": (0, 1, 1), "accelerometer": (1, 3, 0), "velocimeter": (2, 3, 0), "gyro": (3, 3, 0), "rangefinder": (7, 1, 1),
            "jointpos": (9, 1, 0), "jointvel": (10, 1, 0), "framepos": (26, 3, 0), "framequat": (27, 4, 3), "framexaxis": (28, 3, 2),
            "frameyaxis": (29, 3, 2), "framezaxis": (30, 3, 2), "framelinvel": (31, 3, 0), "frameangvel": (32, 3, 0)}
    OBJ = {"body": 1, "xbody": 2, "joint": 3, "geom": 5, "site": 6}

    def __init__(self, xml_text):
        root = ET.fromstring(xml_text)
        els = list(root.find("sensor")) if root.find("sensor") is not None else []
        bare = re.sub(r"<sensor>.*?</sensor>", "", xml_text, flags=re.S)
        self.ref = r = RefModel(bare)
        names = {"site": [x["name"] for x in r.sites], "joint": [x["name"] for x in r.joints], "geom": [x["name"] for x in r.geoms],
                 "body": [x["name"] for x in r.bodies]}
        names["xbody"] = names["body"]
        f = {k: [] for k in FIELDS}
        adr = 0
        for el in els:
            t, dim, dt = self.TAGS[el.tag]
            if el.tag in ("touch", "accelerometer", "rangefinder", "gyro", "velocimeter"):
                kind, obj = "site", el.get("site")
            elif el.tag in ("jointpos", "jointvel"):
                kind, obj = "joint", el.get("joint")
            else:
                kind, obj = el.get("objtype"), el.get("objname")
            for k, v in zip(FIELDS, (t, self.OBJ[kind], names[kind].index(obj), adr, dim, dt, float(el.get("cutoff", 0)))):
                f[k].append(v)
            adr += dim
        self.f = {k: np.asarray(v, dtype=np.float64 if k == "sensor_cutoff" else np.int64) for k, v in f.items()}
        self.legacy = [i for i, el in enumerate(els) if _legacy(el)]
        for el in [el for el in els if not _legacy(el)]:
            root.find("sensor").remove(el)
        self.oracle_model = L.Model(ET.tostring(root, encoding="unicode"))
        lf = self.oracle_model.fields
        self.legacy_adr = [(int(self.f["sensor_adr"][i]), int(lf["sensor_adr"][k]), int(self.f["sensor_dim"][i]))
                           for k, i in enumerate(self.legacy)]
        self.nsensordata = adr

    def sim(self):
        return OracleSim(self.oracle_model.blob)

    def _jac(self, sim, body, point):
        """world-frame point Jacobian (3 x nv each: translation, rotation) from the oracle's body frames"""
        r, nv = self.ref, self.ref.nv
        xpos, xmat = sim.array("xpos").reshape(-1, 3), sim.array("xmat").reshape(-1, 3, 3)
        jp, jr = np.zeros((3, nv)), np.zeros((3, nv))
        b = body
        while b > 0:
            js = r.bodies[b]["joints"]
            assert len(js) <= 1, "the reference handles one joint per body"
            for ji in js:
                j, d = r.joints[ji], r.joints[ji]["dadr"]
                if j["type"] == 0:       # free: world translations, rotations about the body's axes
                    jp[:, d:d + 3] = np.eye(3)
                    for k in range(3):
                        w = xmat[b][:, k]
                        jr[:, d + 3 + k], jp[:, d + 3 + k] = w, np.cross(w, point - xpos[b])
                elif j["type"] == 3:     # hinge: the axis and the anchor ride on the body after its joint
                    w = xmat[b] @ j["axis"]
                    jr[:, d], jp[:, d] = w, np.cross(w, point - (xpos[b] + xmat[b] @ j["pos"]))
                else:                    # slide
                    jp[:, d] = xmat[b] @ j["axis"]
            b = r.bodies[b]["parent"]
        return jp, jr

    def frame(self, sim, i):
        """(body, world point, world rotation) of sensor i's object, from the oracle's kinematics"""
        ot, oid, r = int(self.f["sensor_objtype"][i]), int(self.f["sensor_objid"][i]), self.ref
        if ot == 6:
            return r.sites[oid]["body"], sim.array("site_xpos")[3 * oid:3 * oid + 3], sim.array("site_xmat")[9 * oid:9 * oid + 9].reshape(3, 3)
        if ot == 5:
            return r.geoms[oid]["body"], sim.array("geom_xpos")[3 * oid:3 * oid + 3], sim.array("geom_xmat")[9 * oid:9 * oid + 9].reshape(3, 3)
        R = sim.array("xmat")[9 * oid:9 * oid + 9].reshape(3, 3)
        if ot == 1:
            return oid, sim.array("xipos")[3 * oid:3 * oid + 3], R @ quat2mat(self.oracle_model.fields["body_iquat"][4 * oid:4 * oid + 4])
        return oid, sim.array("xpos")[3 * oid:3 * oid + 3], R

    def values(self, sim):
        """sensor values of the state the oracle's last forward pass saw: (sensordata with NaN in the legacy and framequat
        slots, {sensor: world rotation} of the frame sensors).  Call right after sim.forward()."""
        sd, mats = np.full(self.nsensordata, np.nan), {}
        qpos, qvel = sim.qpos.copy(), sim.qvel.copy()
        for i in range(len(self.f["sensor_type"])):
            if i in self.legacy:
                continue
            t, adr, cut = int(self.f["sensor_type"][i]), int(self.f["sensor_adr"][i]), float(self.f["sensor_cutoff"][i])
            if t in (T["jointpos"], T["jointvel"]):
                j = self.ref.joints[int(self.f["sensor_objid"][i])]
                out = np.array([qpos[j["qadr"]] if t == T["jointpos"] else qvel[j["dadr"]]])
            else:
                b, p, R = self.frame(sim, i)
                p, R = p.copy(), R.copy()   # the oracle's arrays are live views of its state
                mats[i] = R
                jp, jr = self._jac(sim, b, p)
                w, v = jr @ qvel, jp @ qvel
                out = {T["framepos"]: p, T["framelinvel"]: v, T["frameangvel"]: w, T["gyro"]: R.T @ w, T["velocimeter"]: R.T @ v,
                       T["framexaxis"]: R[:, 0], T["frameyaxis"]: R[:, 1], T["framezaxis"]: R[:, 2]}.get(t)
                if out is None:   # framequat: compared through its rotation
                    continue
            if cut > 0 and int(self.f["sensor_datatype"][i]) == 0:
                out = np.clip(out, -cut, cut)
            sd[adr:adr + len(out)] = out
        return sd, mats

    def fill_legacy(self, sd, sim):
        for full, leg, dim in self.legacy_adr:
            sd[full:full + dim] = sim.sensordata[leg:leg + dim]
        return sd

    def step(self, sim, skip=1):
        """`skip` oracle steps; the sensors of the last one (its forward pass sees the state before its integration)"""
        for _ in range(skip - 1):
            sim.step()
        sim.forward()
        sd, mats = self.values(sim)
        sim.step()
        return self.fill_legacy(sd, sim), mats


def assert_sensors(model, got, ref_sd, ref_mats, tag):
    """every sensor of `got` (fp32 sensordata) against the reference values / object rotations"""
    f = model.fields
    for i in range(model.nsensor):
        t, adr, dim = int(f["sensor_type"][i]), int(f["sensor_adr"][i]), int(f["sensor_dim"][i])
        if t == T["framequat"]:
            q = np.asarray(got[adr:adr + 4], float)
            assert abs(np.linalg.norm(q) - 1) < 1e-5, (tag, i)
            assert rel_err(quat2mat(q), ref_mats[i]) < RTOL, (tag, i)
        else:
            tol = ACC_TOL if t in (T["touch"], T["accelerometer"]) else RTOL
            assert not np.isnan(ref_sd[adr:adr + dim]).any(), (tag, i)
            assert rel_err(got[adr:adr + dim], ref_sd[adr:adr + dim]) < tol, (tag, i, got[adr:adr + dim], ref_sd[adr:adr + dim])


def oracle_states(sref, tables, agents, fj, n, stride, settle, seed=0, skip=1):
    """pre-step states along an oracle rollout with random actions, and the reference sensors after `skip` more steps"""
    sim = sref.sim()
    rng = np.random.default_rng(seed)
    n_phys = len(tables.act_space[agents[0]]["low"])

    def act():
        a = {ag: rng.uniform(-1, 1, n_phys) for ag in agents}
        for ag in agents:
            (sim.qvel if fj else sim.ctrl)[tables.agents_action_index[ag]] = a[ag]
        return np.stack([a[ag] for ag in agents])
    for _ in range(settle):
        act(); sim.step()
    out = []
    for _ in range(n):
        for _ in range(stride):
            act(); sim.step()
        pre = (sim.qpos.copy(), sim.qvel.copy(), sim.qacc_warmstart.copy(), sim.ctrl.copy())
        a = act()   # applied once per env step, as the kernel does
        sd, mats = sref.step(sim, skip)
        out.append((pre, a, sd, mats, sim.qpos.copy()))
    return out


def sim_set(sim, model, pre):
    sim.reset()
    sim.qpos[:] = pre[0]; sim.qvel[:] = pre[1]; sim.qacc_warmstart[:] = pre[2]
    if model.nu:
        sim.ctrl[:] = pre[3]


# ---------------------------------------------------------------------------------------------------------------------
# compiler
SMALL = """<mujoco><worldbody><geom name="floor" type="plane" size="5 5 1"/>
  <body name="b" pos="0 0 1"><joint name="h" type="hinge" axis="0 1 0"/><joint name="s" type="slide" axis="1 0 0"/>
   <geom name="g" type="box" size="0.1 0.2 0.3" pos="0.1 0 0"/><site name="t" pos="0 0.1 0"/></body>
  <body name="f" pos="1 0 1"><freejoint name="fj"/><geom type="sphere" size="0.1"/></body>
 </worldbody><sensor>{}</sensor></mujoco>"""
ONE = {"gyro": '<gyro site="t" cutoff="2"/>', "velocimeter": '<velocimeter site="t"/>', "jointpos": '<jointpos joint="h"/>',
       "jointvel": '<jointvel joint="s" cutoff="0.5"/>'}
for _tag in ("framepos", "framequat", "framelinvel", "frameangvel", "framexaxis", "frameyaxis", "framezaxis"):
    for _ot, _on in (("site", "t"), ("body", "b"), ("xbody", "b"), ("geom", "g"), ("xbody", "world"), ("geom", "floor")):
        ONE[f"{_tag}-{_ot}-{_on}"] = f'<{_tag} objtype="{_ot}" objname="{_on}" noise="0.1" user="1 2"/>'


@pytest.mark.parametrize("key", sorted(ONE))
def test_compiler_matches_independent_derivation(key):
    xml = SMALL.format(ONE[key] + '<touch site="t"/>')
    model, ref = L.Model(xml), SensorRef(xml)
    for name in FIELDS:
        assert np.array_equal(np.asarray(model.fields[name]), ref.f[name]), (key, name, model.fields[name], ref.f[name])


@pytest.mark.parametrize("name", sorted(LEVELS_IMU))
def test_fixture_sensor_fields(name):
    text = level_text(name)
    model, ref = L.Model(text), SensorRef(text)
    for f in FIELDS:
        assert np.array_equal(np.asarray(model.fields[f]), ref.f[f]), (name, f)
    assert set(np.asarray(model.fields["sensor_objtype"]).tolist()) >= ({1, 2, 5, 6} if name == "box_imu" else {3, 5, 6})


def test_sensor_datatypes_and_ids():
    xml = SMALL.format('<gyro site="t"/><framequat objtype="body" objname="b"/><framexaxis objtype="geom" objname="g"/>'
                       '<jointpos joint="h"/>')
    f = L.Model(xml).fields
    assert list(f["sensor_type"]) == [3, 27, 28, 9]
    assert list(f["sensor_datatype"]) == [L.DATA_REAL, L.DATA_QUATERNION, L.DATA_AXIS, L.DATA_REAL]
    assert list(f["sensor_objtype"]) == [L.OBJ_SITE, L.OBJ_BODY, L.OBJ_GEOM, L.OBJ_JOINT]
    assert list(f["sensor_dim"]) == [3, 4, 3, 1] and list(f["sensor_adr"]) == [0, 3, 7, 10]


REFUSED = {
    "reftype": ('<framepos name="rp" objtype="site" objname="t" reftype="body" refname="b"/>', "rp"),
    "camera": ('<framepos name="cam" objtype="camera" objname="t"/>', "cam"),
    "free": ('<jointpos name="jp" joint="fj"/>', "jp"),
    "freevel": ('<jointvel name="jv" joint="fj"/>', "jv"),
    "unknown": ('<framequat name="uq" objtype="body" objname="nope"/>', "uq"),
    "unknown_site": ('<gyro name="ug" site="nope"/>', "ug"),
    "unknown_joint": ('<jointpos name="uj" joint="nope"/>', "uj"),
}
for _tag in ("magnetometer", "force", "torque", "subtreecom", "subtreelinvel", "subtreeangmom", "actuatorpos", "actuatorvel",
             "actuatorfrc", "ballquat", "ballangvel", "jointlimitpos", "jointlimitvel", "jointlimitfrc", "tendonpos", "tendonvel",
             "tendonlimitpos", "framelinacc", "frameangacc"):
    REFUSED[_tag] = (f'<{_tag} site="t"/>', f"<{_tag}")


@pytest.mark.parametrize("key", sorted(REFUSED))
def test_refusals_name_the_element(key):
    el, named = REFUSED[key]
    with pytest.raises(Exception, match=named):
        L.Model(SMALL.format(el))


# ---------------------------------------------------------------------------------------------------------------------
# oracle closed forms (zero gravity)
ARM = """<mujoco><option gravity="0 0 0"/><worldbody>
  <body name="arm" pos="0.2 0.1 0.5"><joint name="h" type="hinge" axis="0 0 1"/>
   <geom name="rod" type="capsule" fromto="0 0 0 0.6 0 0" size="0.05"/>
   <site name="tip" pos="0.5 0 0" euler="30 0 60"/></body></worldbody>
 <sensor><gyro site="tip"/><velocimeter site="tip"/><framelinvel objtype="site" objname="tip"/>
  <frameangvel objtype="site" objname="tip"/><framequat objtype="xbody" objname="arm"/><framepos objtype="site" objname="tip"/>
  <jointpos joint="h"/><jointvel joint="h"/></sensor></mujoco>"""

BOX = """<mujoco><option gravity="0 0 0"/><worldbody>
  <body name="box" pos="0 0 1"><freejoint name="r"/><geom type="box" size="0.3 0.2 0.1"/>
   <geom type="sphere" pos="0.4 0.1 -0.05" size="0.1"/></body></worldbody>
 <sensor><framelinvel objtype="body" objname="box"/><framelinvel objtype="xbody" objname="box"/>
  <framequat objtype="xbody" objname="box"/><frameangvel objtype="body" objname="box"/><framepos objtype="body" objname="box"/>
  <framepos objtype="xbody" objname="box"/></sensor></mujoco>"""


def rotz(a):
    return np.array([[math.cos(a), -math.sin(a), 0], [math.sin(a), math.cos(a), 0], [0, 0, 1]])


def site_R(model, site, R_body):
    return R_body @ quat2mat(model.fields["site_quat"][4 * site:4 * site + 4])


@pytest.mark.parametrize("theta", [0.3, 3.5])
def test_oracle_hinge_arm_closed_form(theta):
    model, sref = L.Model(ARM), SensorRef(ARM)
    sim = sref.sim()
    w = 2.5
    sim.qpos[0], sim.qvel[0] = theta, w
    sim.forward()
    sd, mats = sref.values(sim)
    Rb = rotz(theta)
    o = np.array([0.2, 0.1, 0.5])
    p = o + Rb @ np.array([0.5, 0, 0])
    Rs = site_R(model, 0, Rb)
    om = np.array([0, 0, w])
    assert np.allclose(sd[0:3], Rs.T @ om, atol=1e-12)
    assert np.allclose(sd[3:6], Rs.T @ np.cross(om, p - o), atol=1e-12)
    assert abs(np.linalg.norm(sd[3:6]) - w * 0.5) < 1e-12
    assert np.allclose(sd[6:9], np.cross(om, p - o), atol=1e-12)
    assert np.allclose(sd[9:12], om, atol=1e-12)
    assert np.allclose(mats[4], Rb, atol=1e-12)
    assert np.allclose(sd[16:19], p, atol=1e-12)
    assert sd[19] == theta and sd[20] == w


def box_state(sim):
    q = np.array([-0.6, 0.48, 0.0, 0.64])           # |q| = 1 with w < 0
    sim.qpos[:3] = [0.3, -0.2, 1.1]
    sim.qpos[3:7] = q
    v, wl = np.array([0.4, -0.3, 0.2]), np.array([1.5, -0.7, 2.0])
    sim.qvel[:3], sim.qvel[3:6] = v, wl
    return q, v, wl


def test_oracle_free_box_closed_form():
    model, sref = L.Model(BOX), SensorRef(BOX)
    sim = sref.sim()
    q, v, wl = box_state(sim)
    sim.forward()
    sd, mats = sref.values(sim)
    R = quat2mat(q)
    xpos, xipos = np.array([0.3, -0.2, 1.1]), np.array([0.3, -0.2, 1.1]) + R @ model.fields["body_ipos"][3:6]
    assert np.linalg.norm(model.fields["body_ipos"][3:6]) > 0.02
    w = R @ wl
    assert np.allclose(sd[0:3], v + np.cross(w, xipos - xpos), atol=1e-12)
    assert np.allclose(sd[3:6], v, atol=1e-12)
    assert np.allclose(mats[2], R, atol=1e-12)
    assert np.allclose(sd[10:13], w, atol=1e-12)
    assert np.allclose(sd[13:16], xipos, atol=1e-12) and np.allclose(sd[16:19], xpos, atol=1e-12)


def test_oracle_joint_sensors_report_the_pre_step_state():
    sref = SensorRef(ARM)
    sim = sref.sim()
    sim.qpos[0], sim.qvel[0] = 0.7, -1.3
    sd, _ = sref.step(sim)
    assert sd[19] == 0.7 and sd[20] == -1.3
    assert sim.qpos[0] != 0.7


def test_oracle_cutoff_clamps_real_values_only():
    xml = ARM.replace('<gyro site="tip"/>', '<gyro site="tip" cutoff="0.1"/>').replace(
        '<framelinvel objtype="site" objname="tip"/>', '<framelinvel objtype="site" objname="tip" cutoff="0.2"/>').replace(
        '<jointpos joint="h"/>', '<jointpos joint="h" cutoff="0.1"/><framexaxis objtype="xbody" objname="arm" cutoff="0.01"/>')
    sref = SensorRef(xml)
    sim = sref.sim()
    sim.qpos[0], sim.qvel[0] = 1.0, 3.0
    sim.forward()
    sd, _ = sref.values(sim)
    assert np.abs(sd[0:3]).max() <= 0.1 and np.isclose(np.abs(sd[0:3]).max(), 0.1)
    assert np.abs(sd[6:9]).max() <= 0.2 + 1e-15 and np.isclose(np.abs(sd[6:9]).max(), 0.2)
    assert sd[19] == 0.1
    assert np.allclose(sd[20:23], rotz(1.0)[:, 0], atol=1e-12)    # the axis is not clamped


# ---------------------------------------------------------------------------------------------------------------------
# the device code on the SIMT emulator
def emu_forward(xml, qpos, qvel, reverse=False):
    model = L.Model(xml)
    spec, keep = E.simple_spec(model, [], [], 0)
    eb = E.EmuBatch(model.blob, spec, 1, keep)
    eb.qpos[0, :model.nq], eb.qvel[0, :model.nv] = qpos, qvel
    eb.run(E.MODE_PHYSICS, 1, reverse=reverse)
    return model, eb.sensordata[0, :model.nsensordata].astype(np.float64)


@pytest.mark.parametrize("reverse", [False, True])
def test_emulator_quaternion_sign_and_closed_forms(reverse):
    # a hinge beyond pi reports w < 0
    theta = 3.5
    model, sd = emu_forward(ARM, [theta], [2.5], reverse)
    assert np.allclose(sd[12:16], [math.cos(theta / 2), 0, 0, math.sin(theta / 2)], atol=1e-6) and sd[12] < 0
    assert abs(sd[19] - theta) < 1e-6 and abs(sd[20] - 2.5) < 1e-6
    assert np.allclose(sd[9:12], [0, 0, 2.5], atol=1e-5)
    # a free quaternion with w < 0 keeps its sign
    model, sref = L.Model(BOX), SensorRef(BOX)
    sim = sref.sim()
    q, v, wl = box_state(sim)
    _, sd = emu_forward(BOX, sim.qpos.copy(), sim.qvel.copy(), reverse)
    assert np.allclose(sd[6:10], q, atol=1e-6) and sd[6] < 0
    sim.forward()
    assert_sensors(model, sd, *sref.values(sim), "box")


def emu_against_oracle(name, pack, reverse, settle, seed, n=12, skip=1):
    model, tables, agents, fj = load(name)
    spec, keep = make_spec(model, tables, agents, fj, skip_frames=skip)
    if not pack:
        spec.flags |= L.SPEC_NO_PACK
    states = oracle_states(SensorRef(level_text(name)), tables, agents, fj, n, stride=3, settle=settle, seed=seed, skip=skip)
    eb = E.EmuBatch(model.blob, spec, n, keep)
    for e, (pre, a, _, _, _) in enumerate(states):
        eb.qpos[e, :model.nq], eb.qvel[e, :model.nv], eb.warmstart[e, :model.nv] = pre[0], pre[1], pre[2]
        if model.nu:
            eb.ctrl[e, :model.nu] = pre[3]
        eb.actions[e, :, :spec.n_phys_act] = a
    eb.run(E.MODE_PHYSICS, skip, reverse=reverse)
    for e, (_, _, sd, xm, qpos) in enumerate(states):
        assert rel_err(eb.qpos[e, :model.nq], qpos) < RTOL * skip, (name, e)
        assert_sensors(model, eb.sensordata[e, :model.nsensordata], sd, xm, (name, e))
    return eb


@pytest.mark.parametrize("reverse", [False, True])
@pytest.mark.parametrize("settle,seed", [(0, 1), (60, 2)])
@pytest.mark.parametrize("name,pack", [("box_imu", True), ("box_imu", False), ("two_ants_imu", True), ("ant_rk4_imu", True)])
def test_emulator_against_oracle(name, pack, reverse, settle, seed):
    emu_against_oracle(name, pack, reverse, settle, seed)


def test_emulator_skip_frames_5():
    emu_against_oracle("box_imu", True, False, 20, 4, skip=5)


def test_emulator_lane_orders_agree_bitwise():
    a = emu_against_oracle("box_imu", True, False, 30, 5)
    b = emu_against_oracle("box_imu", True, True, 30, 5)
    assert np.array_equal(a.sensordata, b.sensordata)


# ---------------------------------------------------------------------------------------------------------------------
# observation tables
def test_tables_spaces_ownership_and_index():
    model, tables, agents, _ = load("two_ants_imu")
    f = model.fields
    names = [model.id2name(L.OBJ_SENSOR, i) for i in range(model.nsensor)]
    for agent in agents:
        idx = tables.agents_observation_index[agent]["sensors"]
        mine = [i for i, n in enumerate(names) if n.startswith(agent)]
        want = [int(f["sensor_adr"][i]) + k for i in mine for k in range(int(f["sensor_dim"][i]))]
        assert idx == want, agent                                   # sensor-id order
        sp = tables.obs_space[agent]
        lo, hi = sp["low"][:len(idx)], sp["high"][:len(idx)]
        k = 0
        for i in mine:
            d, t = int(f["sensor_dim"][i]), int(f["sensor_type"][i])
            if t == T["framequat"]:
                assert lo[k:k + d] == [-1] * 4 and hi[k:k + d] == [1] * 4
            elif t == T["rangefinder"]:
                assert lo[k:k + d] == [-1] and hi[k:k + d] == [20.0]
            else:
                assert lo[k:k + d] == [-math.inf] * d and hi[k:k + d] == [math.inf] * d
            k += d
    # box_imu: the pillar's sensors belong to nobody, cutoffs bound their slots
    model, tables, agents, _ = load("box_imu")
    names = [model.id2name(L.OBJ_SENSOR, i) for i in range(model.nsensor)]
    idx = tables.agents_observation_index["receiver"]["sensors"]
    owned = {names[i] for i in range(model.nsensor) if int(model.fields["sensor_adr"][i]) in idx}
    assert owned == {n for n in names if not n.startswith("pillar")}
    sp = tables.obs_space["receiver"]
    i = names.index("imu_gyro_cut")
    k = idx.index(int(model.fields["sensor_adr"][i]))
    assert sp["low"][k:k + 3] == [-0.5] * 3 and sp["high"][k:k + 3] == [0.5] * 3


@pytest.mark.parametrize("name", ["box_imu", "two_ants_imu"])
def test_emulator_obs_is_the_gather_of_sensordata(name):
    model, tables, agents, fj = load(name)
    spec, keep = make_spec(model, tables, agents, fj)
    n = 6
    eb = E.EmuBatch(model.blob, spec, n, keep)
    eb.run(E.MODE_RESET)
    rng = np.random.default_rng(3)
    for _ in range(3):
        eb.actions[:, :, :spec.n_phys_act] = rng.uniform(-1, 1, (n, len(agents), spec.n_phys_act))
        eb.run(E.MODE_STEP)
    for a, agent in enumerate(agents):
        idx = tables.agents_observation_index[agent]["sensors"]
        assert len(idx) > 0
        assert np.array_equal(eb.obs[:, a, :len(idx)], eb.sensordata[:, idx])


# ---------------------------------------------------------------------------------------------------------------------
# GPU
def _gpu_batch(name, N, pack, skip):
    import torch
    from mujoco_rl_environment_wrapper_b200.batch import Batch
    model, tables, agents, fj = load(name)
    spec, keep = make_spec(model, tables, agents, fj, skip_frames=skip)
    if not pack:
        spec.flags |= L.SPEC_NO_PACK
    return torch, model, tables, agents, fj, spec, Batch(model, spec, N, keepalive=keep)


@pytest.mark.gpu
@pytest.mark.parametrize("skip", [1, 5])
@pytest.mark.parametrize("name,pack", [("box_imu", True), ("box_imu", False), ("two_ants_imu", True), ("two_ants_imu", False),
                                       ("ant_rk4_imu", True), ("ant_rk4_imu", False)])
def test_gpu_strided_subset_against_oracle(name, pack, skip):
    N = 4096
    torch, model, tables, agents, fj, spec, b = _gpu_batch(name, N, pack, skip)
    nq, nv, nu, ns, n_phys, A = model.nq, model.nv, model.nu, model.nsensordata, spec.n_phys_act, len(agents)
    g = torch.Generator(device="cuda"); g.manual_seed(7)
    b.reset()
    for _ in range(20 // skip + 2):
        b.actions[:, :, :n_phys] = torch.rand((N, A, n_phys), generator=g, device="cuda") * 2 - 1
        b.physics(skip)
    b.sync()
    sub = np.unique(np.concatenate([np.arange(0, N, N // 24), [1, 2, 3, N - 1]]))
    pre = {k: getattr(b, k)[sub].cpu().numpy().astype(np.float64) for k in ("qpos", "qvel", "warmstart", "ctrl")}
    act = torch.rand((N, A, n_phys), generator=g, device="cuda") * 2 - 1
    b.actions[:, :, :n_phys] = act
    act_np = act[sub].cpu().numpy().astype(np.float64)
    b.physics(skip); b.sync()
    sens, q = b.sensordata[sub].cpu().numpy(), b.qpos[sub].cpu().numpy()
    sref = SensorRef(level_text(name))
    sim = sref.sim()
    for i, e in enumerate(sub):
        sim_set(sim, model, (pre["qpos"][i, :nq], pre["qvel"][i, :nv], pre["warmstart"][i, :nv], pre["ctrl"][i, :nu]))
        for a, agent in enumerate(agents):
            (sim.qvel if fj else sim.ctrl)[tables.agents_action_index[agent]] = act_np[i, a]
        sd, mats = sref.step(sim, skip)
        assert rel_err(q[i, :nq], sim.qpos) < RTOL * skip, (name, int(e))
        assert_sensors(model, sens[i, :ns], sd, mats, (name, int(e)))


def _env(N, **kw):
    from mujoco_rl_environment_wrapper_b200 import plugins as P
    from mujoco_rl_environment_wrapper_b200.mujoco_rl import MuJoCoRL
    cfg = {"xmlPath": os.path.join(SENSOR_LEVELS, "two_ants_imu.xml"), "infoJson": os.path.join(LEVELS, "info_2A.json"),
           "agents": ["sender", "receiver"], "num_envs": N, "seed": 3, "environmentDynamics": [P.Language],
           "rewardFunctions": [P.tag_distance_reward], "doneFunctions": [P.distance_done]}
    cfg.update(kw)
    return MuJoCoRL(cfg)


@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 8])
def test_gpu_python_api(N):
    import torch
    env = _env(N)
    env.reset()
    act = {a: torch.zeros((N, 9)) if N > 1 else np.zeros(9) for a in env.agents}
    env.step(act)
    m = env.model.sensor("sender_framequat")
    assert int(m.type[0]) == T["framequat"] and int(m.dim[0]) == 4 and int(m.objtype[0]) == L.OBJ_SITE
    assert int(m.objid[0]) == env.model.name2id(L.OBJ_SITE, "sender_imu") and float(m.cutoff[0]) == 0
    j = env.model.sensor("receiver_hip_1_vel")
    assert int(j.objtype[0]) == L.OBJ_JOINT and int(j.objid[0]) == env.model.name2id(L.OBJ_JOINT, "hip_1_2")
    d = env.data.sensor("sender_framequat").data
    sd = env.data.sensordata
    adr = int(m.adr[0])
    if N == 1:
        assert isinstance(d, np.ndarray) and d.shape == (4,) and np.array_equal(d, sd[adr:adr + 4])
    else:
        assert tuple(d.shape) == (N, 4) and torch.equal(d, sd[:, adr:adr + 4])
    q = d if N == 1 else d.cpu().numpy()
    assert np.allclose(np.linalg.norm(np.reshape(q, (-1, 4)), axis=1), 1, atol=1e-5)
    for agent in env.agents:
        sp = env.observation_space(agent)
        sdat = env.get_sensor_data(agent)
        k = len(env.agents_observation_index[agent]["sensors"])
        assert k == 2 * 0 + 1 + 3 + 3 + 3 + 4 + 4 + 3
        lo, hi = np.asarray(sp.low[:k]), np.asarray(sp.high[:k])
        s = np.asarray(sdat.cpu() if torch.is_tensor(sdat) else sdat).reshape(-1, k)
        assert (s >= lo - 1e-6).all() and (s <= hi + 1e-6).all()
        assert np.isinf(hi).sum() == k - 1 - 4 and (hi[lo == -1] == 1).sum() == 4


@pytest.mark.gpu
def test_gpu_autoreset_new_sensors_equal_step_then_reset():
    """the new sensors in final_observation and in the next episode's first observation equal a plain step followed by
    reset(mask) (only the physics slots: the reset's drawn Language action differs by design)"""
    import torch
    N = 64
    auto, plain = _env(N, autoReset=True, maxSteps=5), _env(N, maxSteps=5)
    for e in (auto, plain):
        e.reset()
    g = torch.Generator(device=auto.device).manual_seed(1)
    scale, shift = torch.tensor([2.0] * 8 + [3.0], device=auto.device), torch.tensor([1.0] * 8 + [0.0], device=auto.device)
    seen = 0
    for t in range(12):
        act = torch.rand((N, 2, 9), generator=g, device=auto.device) * scale - shift
        oa, _, _, _, ia = auto.step(act)
        op, _, tp, trp, _ = plain.step(act)
        done = (tp["__all__"] | trp["__all__"]).to(auto.device).bool()
        for a in auto.agents:
            k = len(auto.agents_observation_index[a]["sensors"])
            fin = ia[a]["_final_observation"].to(auto.device)
            assert torch.equal(fin, done)
            assert torch.equal(ia[a]["final_observation"][fin][:, :k], op[a][fin][:, :k])
        if bool(done.any()):
            seen += 1
            plain.reset(mask=done)
            for a in auto.agents:
                k = len(auto.agents_observation_index[a]["sensors"])
                assert torch.equal(auto.get_observations(a)[done][:, :k], plain.get_observations(a)[done][:, :k])
        assert torch.equal(auto.batch.sensordata, plain.batch.sensordata)
        assert torch.equal(auto.batch.qpos, plain.batch.qpos)
    assert seen >= 2


@pytest.mark.gpu
def test_gpu_65536_envs_two_ants_imu_stays_finite():
    import torch
    N = 65536
    torch_, model, tables, agents, fj, spec, b = _gpu_batch("two_ants_imu", N, True, 1)
    g = torch.Generator(device="cuda"); g.manual_seed(2)
    b.reset()
    for _ in range(50):
        b.actions[:, :, :spec.n_phys_act] = torch.rand((N, len(agents), spec.n_phys_act), generator=g, device="cuda") * 2 - 1
        b.physics(1)
    b.sync()
    sd = b.sensordata[:, :model.nsensordata]
    assert torch.isfinite(sd).all() and torch.isfinite(b.qpos).all()
    assert float(sd.abs().max()) > 0
