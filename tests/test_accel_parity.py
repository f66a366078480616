"""The step kernel's accelerations against the fp64 oracle, not only the state after one step.

With h = 0.002 an acceleration reaches the state only as h * qacc in qvel and h^2 * qacc in qpos, so the one-step state
check of test_emu_parity / test_gpu_parity (rtol 1e-4) pins the dynamics to about 0.5 % of the acceleration: a kernel
whose body masses are 0.2 % off, or whose joint damping is 1 % off, passes it.  Here, from oracle rollout states of every
scene (plus states where the two ants' trees are coupled by contacts, and states next to a wall), the kernel is compared
at the level of accelerations:

1. solver acceleration: `forward` from (qpos, qvel, ctrl) leaves the solver's qacc in `warmstart`; against the oracle's
   qacc after `forward()` from the same state,
       |dqacc|_inf <= TAU_A * max(|qacc|_inf, g)   and   |dqacc|_M <= TAU_M * |qacc|_M   (M: the oracle's mass matrix);
2. effective acceleration of one `physics(1)` step (implicit damping `(M + hD) a' = ...`, RK4's stage-weighted
   increment), as the velocity increment from the pre-step velocity after the action overwrite:
       |dv_kernel - dv_oracle|_inf <= TAU_DV * max(|dv_oracle|_inf, h g);
3. coverage: the sample holds active joint-limit rows, multi-contact states, contacts coupling the two ants' trees, every
   copy of a packed warp with a ragged env count, and box-box / capsule-box contacts where a level has boxes;
4. power: the checks flag model blobs with masses x 1.002, dof damping x 1.01, pair friction x 1.01 and pair solref x 1.01
   (the first two pass the 1e-4 state check), and a solver cut to one Newton iteration (MJB_SOLVER_ITERS=1);
5. far from the origin: the free roots of a level whose only static geometry is the floor translated by 10, 100, 1000 m.

Tolerances: the worst value observed over the full sample of every scene, times about 4 (emulator) and 3.5 (B200):
    emulator (kernel source on the host, IEEE fp32):   |dqacc|/scale 1.7e-5, M-norm 1.5e-5, dv 1.9e-5 (all on 3S)
    B200 (sm_100a, --use_fast_math; 1000 W limit):      |dqacc|/scale 2.8e-5, M-norm 2.9e-5, dv 3.0e-5 (all on 3S)
The B200's floor is about 1.7x the emulator's (fast-math), so each side keeps its own constants.  The perturbations sit
2x (masses, on 2A) to 300x (pair solref) above them; one Newton iteration, 10^3 to 10^4x.
Far from the origin (1A, |dqacc|/scale, emulator / B200): 0 m 2.8e-6 / 1.1e-5, 10 m 3.1e-6 / 1.1e-5, 100 m 1.7e-5 /
2.7e-5, 1000 m 2.1e-4 / 2.1e-4.  The error grows with ulp(x) of the fp32 root position; the levels' arenas lie within
+-10 m, where TAU_A holds with room to spare."""
import copy
import functools

import numpy as np
import pytest

import emu_harness as E
from common import load_scene, make_spec, oracle_states
from mujoco_rl_environment_wrapper_b200 import _lib as L

G = 9.81
RTOL_STATE = 1e-4                                   # the one-step state check of test_emu_parity / test_gpu_parity
TAU_A, TAU_M, TAU_DV = 8e-5, 6e-5, 8e-5             # emulator
TAU_A_GPU, TAU_M_GPU, TAU_DV_GPU = 1e-4, 1e-4, 1e-4  # B200
SENTINEL = 0.6180339                                # actions that forward mode must not scatter

# scene: (n, stride, settle) of a rollout from qpos0, and of a rollout started next to the wall `border5` (levels
# with boxes), or None.  Counts are ragged for the packed scenes (K = 2 for one ant, 4 for a free box).
SAMPLES = {
    "2A": ((24, 25, 150), (8, 15, 60)),
    "C1": ((15, 20, 100), (8, 15, 60)),
    "1A": ((11, 20, 40), None),
    "S1": ((10, 10, 50), (11, 10, 20)),
    "S2": ((10, 10, 50), (11, 10, 20)),
    "S3": ((10, 10, 50), (11, 10, 20)),
    "S4": ((10, 10, 50), (11, 10, 20)),
    "3S": ((8, 30, 150), (6, 15, 60)),
}
# the busiest state of each scene's sample holds at least this many contacts
MIN_BUSIEST = {"2A": 4, "C1": 3, "1A": 3, "S1": 4, "S2": 4, "S3": 4, "S4": 4, "3S": 3}


def pack_factor(model, n):
    """envs per warp (csrc/dev_model_build.h, choose_pack)"""
    return max(1, min(32 // max(1, model.nv), 4, n))


# ---- sample and fp64 reference ------------------------------------------------------------------------------------
def next_to_wall(model):
    """start(qpos) for oracle_states: the first free root just off the +x face of the static box `border5`"""
    from oracle import OracleSim
    g = model.name2id(L.OBJ_GEOM, "border5_geom")
    sim = OracleSim(model.blob)
    sim.forward()
    face = sim.geom_xpos[g][0] + model.fields["geom_size"].reshape(-1, 3)[g][0]
    root_body = int(model.fields["jnt_bodyid"][0])
    root_geom = int(np.flatnonzero(model.fields["geom_bodyid"] == root_body)[0])
    reach = 0.5 if int(model.fields["geom_type"][root_geom]) == 6 else 0.75   # box half-size / an ant's legs in x

    def start(qpos):
        qpos[0] = face + reach + 0.005
        qpos[1] = sim.geom_xpos[g][1] + 0.5
    return start


def reference(sim, model, pre):
    """the oracle's forward pass and one step from the pre-step state `pre` (as oracle_states returns it)"""
    qpos, qvel, ws, ctrl, _ = pre
    nv = model.nv
    sim.reset()
    sim.qpos[:], sim.qvel[:], sim.qacc_warmstart[:] = qpos, qvel, ws
    if model.nu:
        sim.ctrl[:] = ctrl
    sim.forward()
    r = {"qacc": sim.qacc.copy(), "M": sim.array("M").reshape(nv, nv).copy(), "pairs": sorted(sim.contact_pairs())}
    J = sim.array("efc_J").reshape(-1, nv).copy() if sim.nefc else np.zeros((0, nv))
    force = sim.array("efc_force").copy() if sim.nefc else np.zeros(0)
    nlim = 0            # joint-limit rows come first: one +-1 entry each
    while nlim < len(J) and np.count_nonzero(J[nlim]) == 1 and abs(np.abs(J[nlim]).sum() - 1) < 1e-12:
        nlim += 1
    r["limits"] = int((force[:nlim] > 0).sum())
    sim.step()
    r["qpos"], r["qvel"] = sim.qpos.copy(), sim.qvel.copy()
    return r


def inter_ant_states(model, tables, trials, seed=21):
    """the receiver dropped onto the sender (test_inter_ant_contacts_*): pre-step states every 20 steps"""
    from oracle import OracleSim
    sim = OracleSim(model.blob)
    rng = np.random.default_rng(seed)
    idx = np.array(tables.agents_action_index["sender"] + tables.agents_action_index["receiver"])
    out = []
    for trial in range(trials):
        sim.reset()
        sim.qpos[15:18] = sim.qpos[0:3] + np.array([rng.uniform(-0.3, 0.3), rng.uniform(-0.3, 0.3), 0.45 + 0.2 * rng.random()])
        yaw = rng.uniform(0, np.pi)
        sim.qpos[18:22] = [np.cos(yaw / 2), 0, 0, np.sin(yaw / 2)]
        for t in range(200):
            c = rng.uniform(-1, 1, 16)
            sim.ctrl[idx] = c
            if t >= 60 and t % 20 == 0:
                out.append((sim.qpos.copy(), sim.qvel.copy(), sim.qacc_warmstart.copy(), sim.ctrl.copy(), c.reshape(2, 8).copy()))
            sim.step()
    return out


class Sample:
    """pre-step states of one scene with their fp64 references"""

    def __init__(self, scene, pres):
        from oracle import OracleSim
        self.scene = scene
        self.model, self.tables, self.agents, self.fj = load_scene(scene)
        self.pres = pres
        sim = OracleSim(self.model.blob)
        self.refs = [reference(sim, self.model, p) for p in pres]

    @classmethod
    def build(cls, scene, scale=1):
        model, tables, agents, fj = load_scene(scene)
        plain, wall = SAMPLES[scene]
        n, stride, settle = plain
        pres = [p for p, _ in oracle_states(model, tables, agents, fj, n * scale, stride=stride, settle=settle, seed=3)]
        if wall is not None:
            n, stride, settle = wall
            pres += [p for p, _ in oracle_states(model, tables, agents, fj, n * scale, stride=stride, settle=settle, seed=5,
                                                 start=next_to_wall(model))]
        return cls(scene, pres)

    def with_states(self, pres):
        """the same references for other kernel inputs (e.g. translated copies of the states)"""
        t = copy.copy(self)
        t.pres = pres
        return t

    def spec(self):
        return make_spec(self.model, self.tables, self.agents, self.fj)


@functools.lru_cache(maxsize=None)
def emu_sample(scene):
    if scene == "coupled":
        model, tables, _, _ = load_scene("2A")
        return Sample("2A", inter_ant_states(model, tables, 3))
    return Sample.build(scene)


# ---- kernel runs ---------------------------------------------------------------------------------------------------
def _rows(s):
    m = s.model
    return (np.stack([p[0] for p in s.pres]), np.stack([p[1] for p in s.pres]), np.stack([p[2] for p in s.pres]),
            np.stack([p[3] for p in s.pres]) if m.nu else None, np.stack([p[4] for p in s.pres]))


def run_emu(s, blob=None):
    """forward and physics(1) on the emulator; returns (forward: warmstart, qvel, ctrl; physics: qpos, qvel)"""
    m = s.model
    spec, keep = s.spec()
    qpos, qvel, ws, ctrl, act = _rows(s)
    out = []
    for mode in (E.MODE_FORWARD, E.MODE_PHYSICS):
        eb = E.EmuBatch(m.blob if blob is None else blob, spec, len(s.pres), keep)
        eb.qpos[:, :m.nq], eb.qvel[:, :m.nv], eb.warmstart[:, :m.nv] = qpos, qvel, ws
        if m.nu:
            eb.ctrl[:, :m.nu] = ctrl
        eb.actions[:, :, :spec.n_phys_act] = SENTINEL if mode == E.MODE_FORWARD else act
        eb.run(mode, 1)
        out.append({k: eb.buf[k].astype(np.float64) for k in ("qpos", "qvel", "ctrl", "warmstart", "ncon")})
    return out


def run_gpu(s, model=None):
    """the same through the C-ABI on the GPU (`model`: a perturbed host model of the same scene)"""
    import torch
    from mujoco_rl_environment_wrapper_b200.batch import Batch
    m = s.model if model is None else model
    spec, keep = make_spec(m, s.tables, s.agents, s.fj)
    qpos, qvel, ws, ctrl, act = _rows(s)
    t = lambda a: torch.tensor(a, dtype=torch.float32)
    out = []
    for fwd in (True, False):
        b = Batch(m, spec, len(s.pres), keepalive=keep)
        b.qpos[:, :m.nq], b.qvel[:, :m.nv], b.warmstart[:, :m.nv] = t(qpos), t(qvel), t(ws)
        if m.nu:
            b.ctrl[:, :m.nu] = t(ctrl)
        if fwd:
            b.actions[:, :, :spec.n_phys_act] = SENTINEL
            b.forward()
        else:
            b.actions[:, :, :spec.n_phys_act] = t(act)
            b.physics(1)
        b.sync()
        out.append({k: b.buf[k].cpu().numpy().astype(np.float64) for k in ("qpos", "qvel", "ctrl", "warmstart", "ncon")})
        del b
    return out


# ---- the checks ----------------------------------------------------------------------------------------------------
def rel_err(x, ref):
    return float((np.abs(x - ref) / np.maximum(1.0, np.abs(ref))).max()) if len(ref) else 0.0


def errors(s, fwd, phys):
    """per state: |dqacc|_inf / max(|qacc|_inf, g), M-norm ratio, velocity-increment error, and the old state check"""
    m = s.model
    nq, nv = m.nq, m.nv
    h = m.timestep
    # forward mode scatters no action: ctrl and qvel are what was loaded, bit for bit
    _, qvel0, _, ctrl0, _ = _rows(s)
    assert np.array_equal(fwd["qvel"][:, :nv], qvel0.astype(np.float32).astype(np.float64))
    if m.nu:
        assert np.array_equal(fwd["ctrl"][:, :m.nu], ctrl0.astype(np.float32).astype(np.float64))
    out = {k: np.zeros(len(s.pres)) for k in ("a", "M", "dv", "state")}
    for e, (pre, ref) in enumerate(zip(s.pres, s.refs)):
        a, da = ref["qacc"], fwd["warmstart"][e, :nv] - ref["qacc"]
        out["a"][e] = np.abs(da).max() / max(np.abs(a).max(), G)
        out["M"][e] = np.sqrt(max(da @ ref["M"] @ da, 0.0)) / max(np.sqrt(a @ ref["M"] @ a), 1e-12)
        v0 = pre[1].astype(np.float32).astype(np.float64)
        dv_ref = ref["qvel"] - pre[1]
        out["dv"][e] = np.abs((phys["qvel"][e, :nv] - v0) - dv_ref).max() / max(np.abs(dv_ref).max(), h * G)
        out["state"][e] = max(rel_err(phys["qpos"][e, :nq], ref["qpos"]), rel_err(phys["qvel"][e, :nv], ref["qvel"]))
    return out


def worst(err):
    return {k: float(v.max()) for k, v in err.items()}


def assert_within(s, err, taus, tag=""):
    ta, tm, tdv = taus
    w = worst(err)
    print(f"{tag}{s.scene}: {len(s.pres)} states, |dqacc|/scale {w['a']:.2e}, M-norm {w['M']:.2e}, dv {w['dv']:.2e}, "
          f"state {w['state']:.2e}")
    assert w["a"] <= ta, (s.scene, int(err["a"].argmax()), w)
    assert w["M"] <= tm, (s.scene, int(err["M"].argmax()), w)
    assert w["dv"] <= tdv, (s.scene, int(err["dv"].argmax()), w)
    assert w["state"] < RTOL_STATE, (s.scene, w)


def moving_tree(m):
    """per body: the root body of its kinematic tree, or -1 for a static body"""
    f = m.fields
    root = f["body_rootid"]
    return np.where(f["body_dofnum"][root] > 0, root, -1)


def coverage(s, fwd):
    """what the sample reaches, from the oracle's constraint rows and contacts; the kernel finds the same pairs"""
    m = s.model
    f = m.fields
    gb, gt = f["geom_bodyid"], f["geom_type"]
    tree = moving_tree(m)
    ncon = [len(r["pairs"]) for r in s.refs]
    coupled = sum(any(tree[gb[a]] != tree[gb[b]] and tree[gb[a]] >= 0 and tree[gb[b]] >= 0 for a, b in r["pairs"])
                  for r in s.refs)
    kinds = {tuple(sorted((int(gt[a]), int(gt[b])))) for r in s.refs for a, b in r["pairs"]}
    K = pack_factor(m, len(s.pres))
    contact_copies = {e % K for e, n in enumerate(ncon) if n}
    for e, r in enumerate(s.refs):
        assert int(fwd["ncon"][e]) == len(r["pairs"]), (s.scene, e)
    return {"limits": sum(r["limits"] for r in s.refs), "limit_states": sum(r["limits"] > 0 for r in s.refs),
            "busiest": max(ncon), "contact_states": sum(n > 0 for n in ncon), "coupled": coupled, "kinds": kinds,
            "K": K, "ragged": len(s.pres) % K != 0, "contact_copies": contact_copies}


def assert_coverage(s, cov):
    print(f"{s.scene}: coverage {cov}")
    scene = s.scene
    assert cov["contact_states"] >= 3, cov
    assert cov["busiest"] >= MIN_BUSIEST[scene], cov
    if s.model.nv > 6:
        assert cov["limit_states"] > 0, "the sample must hold active joint-limit rows"
    if cov["K"] > 1:
        assert cov["ragged"] and cov["contact_copies"] == set(range(cov["K"])), cov
    if SAMPLES[scene][1] is not None:       # levels with static boxes
        box = (6, 6) if scene.startswith("S") else (3, 6)     # a free box, or an ant's capsules
        assert box in cov["kinds"], cov


# ---- emulator half -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("scene", list(SAMPLES))
def test_accelerations_match_oracle_emu(scene):
    s = emu_sample(scene)
    fwd, phys = run_emu(s)
    assert_within(s, errors(s, fwd, phys), (TAU_A, TAU_M, TAU_DV), "emu ")
    assert_coverage(s, coverage(s, fwd))


def test_coupled_trees_accelerations_match_oracle_emu():
    """contacts between the two ants' trees: the single 28 x 28 register factorisation"""
    s = emu_sample("coupled")
    fwd, phys = run_emu(s)
    assert_within(s, errors(s, fwd, phys), (TAU_A, TAU_M, TAU_DV), "emu coupled ")
    cov = coverage(s, fwd)
    assert cov["coupled"] >= max(5, len(s.pres) // 6), cov


def patch(blob, name, scale):
    from test_model_params import blob_offsets
    raw = bytearray(blob)
    _, cnt, off = blob_offsets(bytes(raw))[name]
    a = np.frombuffer(raw, np.float64, cnt, off).copy()
    if name == "pair_friction":
        a[0::3] *= scale                    # sliding friction, the coefficient the pyramid uses
    else:
        a *= scale
    assert np.abs(a).max() > 0, name
    raw[off:off + 8 * cnt] = a.tobytes()
    return bytes(raw)


POWER_SCENES = ("2A", "C1", "3S", "S1", "coupled")
GAP_SCENES = ("2A", "3S")          # where a 0.2 % mass / 1 % damping error stays below the state check's 1e-4
PERTURBATIONS = [("body_mass", 1.002), ("dof_damping", 1.01), ("pair_friction", 1.01), ("pair_solref", 1.01)]


def flagged(worsts, taus):
    """names of the checks a perturbed kernel fails"""
    return [k for k, t in zip(("a", "M", "dv"), taus) if worsts[k] > t]


@pytest.mark.parametrize("name,scale", PERTURBATIONS)
def test_power_perturbed_blob_is_flagged_emu(name, scale):
    """the kernel on a perturbed blob, the oracle on the true one: the acceleration checks fail, each by at least two of
    the three measures (so that no single tolerance decides it).  Masses and damping pass the 1e-4 state check on the
    two-ant levels while the acceleration checks of the same states fail: the gap these tests close."""
    w = {"a": 0.0, "M": 0.0, "dv": 0.0, "state": 0.0}
    for scene in POWER_SCENES:
        s = emu_sample(scene)
        if name == "dof_damping" and not s.model.fields["dof_damping"].any():
            continue
        fwd, phys = run_emu(s, patch(s.model.blob, name, scale))
        ws = worst(errors(s, fwd, phys))
        if name in ("body_mass", "dof_damping") and scene in GAP_SCENES:
            assert ws["state"] < RTOL_STATE and len(flagged(ws, (TAU_A, TAU_M, TAU_DV))) >= 2, (scene, ws)
        for k, v in ws.items():
            w[k] = max(w[k], v)
    hits = flagged(w, (TAU_A, TAU_M, TAU_DV))
    print(f"{name} x {scale}: {w} -> {hits}")
    assert len(hits) >= 2, (name, w)


def test_power_one_newton_iteration_is_flagged_emu(monkeypatch):
    """MJB_SOLVER_ITERS=1 (read at batch creation): the contact-rich states are flagged"""
    monkeypatch.setenv("MJB_SOLVER_ITERS", "1")
    w = {"a": 0.0, "M": 0.0, "dv": 0.0}
    for scene in ("2A", "coupled"):
        s = emu_sample(scene)
        fwd, phys = run_emu(s)
        err = errors(s, fwd, phys)
        rich = np.array([len(r["pairs"]) >= 3 for r in s.refs])
        assert rich.sum() >= 3
        for k in w:
            w[k] = max(w[k], float(err[k][rich].max()))
    hits = flagged(w, (TAU_A, TAU_M, TAU_DV))
    print(f"MJB_SOLVER_ITERS=1: {w} -> {hits}")
    assert len(hits) >= 2, w


FAR = (0.0, 10.0, 100.0, 1000.0)


def far_errors(s, fwd_of):
    """|dqacc|/scale per translation: the free roots moved by (d, d/2) m, the oracle at the untranslated state"""
    m = s.model
    roots = [int(m.fields["jnt_qposadr"][j]) for j in range(m.njnt) if int(m.fields["jnt_type"][j]) == L.JNT_FREE]
    out = {}
    for d in FAR:
        pres = []
        for p in s.pres:
            q = p[0].copy()
            for a in roots:
                q[a:a + 2] += [d, d / 2]
            pres.append((q,) + p[1:])
        w = fwd_of(s.with_states(pres))
        out[d] = max(np.abs(w[e, :m.nv] - r["qacc"]).max() / max(np.abs(r["qacc"]).max(), G) for e, r in enumerate(s.refs))
    return out


def test_far_from_origin_emu():
    """1A: the floor plane is the level's only static geom, so the physics is translation-invariant"""
    s = emu_sample("1A")
    static = [g for g in range(s.model.ngeom) if moving_tree(s.model)[s.model.fields["geom_bodyid"][g]] < 0]
    assert [int(s.model.fields["geom_type"][g]) for g in static] == [0]
    err = far_errors(s, lambda t: run_emu(t)[0]["warmstart"])
    print("emu far from origin: " + ", ".join(f"{d:g} m {e:.2e}" for d, e in err.items()))
    assert err[10.0] <= TAU_A, err


# ---- GPU half ------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def gpu_sample(scene):
    if scene == "coupled":
        model, tables, _, _ = load_scene("2A")
        return Sample("2A", inter_ant_states(model, tables, 12))
    return Sample.build(scene, scale=3)


@pytest.mark.gpu
@pytest.mark.parametrize("scene", list(SAMPLES) + ["coupled"])
def test_accelerations_match_oracle_gpu(scene):
    s = gpu_sample(scene)
    fwd, phys = run_gpu(s)
    assert_within(s, errors(s, fwd, phys), (TAU_A_GPU, TAU_M_GPU, TAU_DV_GPU), "gpu ")
    cov = coverage(s, fwd)
    if scene == "coupled":
        assert cov["coupled"] >= max(5, len(s.pres) // 6), cov
    else:
        assert_coverage(s, cov)


@pytest.mark.gpu
def test_power_perturbed_masses_are_flagged_gpu():
    """masses x 1.002 (mjb_model_set_field): flagged by at least two of the three acceleration checks"""
    w = {"a": 0.0, "M": 0.0, "dv": 0.0, "state": 0.0}
    for scene in ("2A", "C1", "3S"):
        s = gpu_sample(scene)
        model, _, _, _ = load_scene(s.scene)
        model.set_field("body_mass", model.fields["body_mass"] * 1.002)
        fwd, phys = run_gpu(s, model)
        for k, v in worst(errors(s, fwd, phys)).items():
            w[k] = max(w[k], v)
    hits = flagged(w, (TAU_A_GPU, TAU_M_GPU, TAU_DV_GPU))
    print(f"gpu body_mass x 1.002: {w} -> {hits}")
    assert len(hits) >= 2, w


@pytest.mark.gpu
def test_far_from_origin_gpu():
    s = gpu_sample("1A")
    err = far_errors(s, lambda t: run_gpu(t)[0]["warmstart"])
    print("gpu far from origin: " + ", ".join(f"{d:g} m {e:.2e}" for d, e in err.items()))
    assert err[10.0] <= TAU_A_GPU, err
