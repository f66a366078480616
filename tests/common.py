"""Shared helpers for the tests: scene configs (SURVEY 8d), EnvSpec construction without a GPU."""
import ctypes
import os

import numpy as np

from mujoco_rl_environment_wrapper_b200 import _lib as L
from mujoco_rl_environment_wrapper_b200.tables import Tables

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LEVELS = os.path.join(ROOT, "tests", "levels")

SCENES = {
    # name: (xml, agents, free_joint)
    "2A": ("two_ants.xml", ["sender", "receiver"], False),
    "1A": ("ant_rk4.xml", ["torso"], False),
    "C1": ("one_ant_arena.xml", ["sender"], False),
    "3S": ("two_ants_touch_acc.xml", ["sender", "receiver"], True),
    "S1": ("box_touch.xml", ["receiver"], True),
    "S2": ("box_accelerometer.xml", ["receiver"], True),
    "S3": ("box_rangefinder.xml", ["receiver"], True),
    "S4": ("box_framexaxis.xml", ["receiver"], True),
}


def load_scene(name):
    xml, agents, fj = SCENES[name]
    path = os.path.join(LEVELS, xml)
    text = open(path).read()
    model = L.Model(text)
    tables = Tables(text, model, agents, fj)
    return model, tables, agents, fj


def make_spec(model, tables, agents, free_joint, skip_frames=1, max_steps=1024, dynamics=(), rewards=(), dones=(),
              targets=(), seed=1234):
    """dynamics: list of (kind, n_act, n_obs, param0); rewards/dones: list of (kind, param0);
    targets: list of (objtype, objid)."""
    A = len(agents)
    spec = L.EnvSpec()
    spec.n_agents, spec.free_joint, spec.skip_frames, spec.max_steps = A, int(free_joint), skip_frames, max_steps
    n_phys = len(tables.act_space[agents[0]]["low"])
    spec.n_phys_act = n_phys
    act_index, obs_index, adr = [], [], [0]
    for a, agent in enumerate(agents):
        act_index += tables.agents_action_index[agent]
        oi = tables.agents_observation_index[agent]
        obs_index += [(0 << 24) | i for i in oi["sensors"]] + [(1 << 24) | i for i in oi["qpos"]] + [(2 << 24) | i for i in oi["qvel"]]
        adr.append(len(obs_index))
        spec.agent_body[a] = tables.agent_body[agent]
    pos, extra_obs = n_phys, 0
    for k, (kind, n_act, n_obs, p0) in enumerate(dynamics):
        p = spec.dynamics[k]
        p.kind, p.act_lo, p.act_hi, p.n_obs = kind, pos, pos + n_act, n_obs
        p.param[0] = p0
        pos += n_act
        extra_obs += n_obs
    for k, (kind, p0) in enumerate(rewards):
        spec.rewards[k].kind = kind
        spec.rewards[k].param[0] = p0
    for k, (kind, p0) in enumerate(dones):
        spec.dones[k].kind = kind
        spec.dones[k].param[0] = p0
    spec.n_dynamics, spec.n_rewards, spec.n_dones = len(dynamics), len(rewards), len(dones)
    spec.act_dim = pos
    for a in range(A):
        spec.obs_dim[a] = adr[a + 1] - adr[a] + extra_obs
    for a in range(A + 1):
        spec.obs_adr[a] = adr[a]
    spec.n_targets = len(targets)
    for t, (ot, oid) in enumerate(targets):
        spec.target_objtype[t], spec.target_objid[t] = ot, oid
    spec.seed = seed
    ai = (ctypes.c_int32 * max(1, len(act_index)))(*act_index)
    oi_ = (ctypes.c_int32 * max(1, len(obs_index)))(*obs_index)
    spec.act_index = ctypes.cast(ai, ctypes.POINTER(ctypes.c_int32))
    spec.obs_index = ctypes.cast(oi_, ctypes.POINTER(ctypes.c_int32))
    return spec, (ai, oi_)


def oracle_states(model, tables, agents, free_joint, n_states, stride=4, seed=0, settle=0, start=None):
    """Pre-step states (qpos, qvel, warmstart, physical action per agent) along an oracle rollout with
    random actions; the rollout itself defines the expected post-step state.  `start(qpos)` may edit the
    initial qpos in place (e.g. to begin next to a wall)."""
    from oracle import OracleSim
    sim = OracleSim(model.blob)
    if start is not None:
        start(sim.qpos)
    rng = np.random.default_rng(seed)
    n_phys = len(tables.act_space[agents[0]]["low"])
    out = []
    for i in range(settle + n_states * stride):
        acts = {a: rng.uniform(-1, 1, n_phys) for a in agents}
        for a in agents:
            idx = tables.agents_action_index[a]
            if free_joint:
                sim.qvel[idx] = acts[a]
            else:
                sim.ctrl[idx] = acts[a]
        if i >= settle and (i - settle) % stride == 0:
            pre = (sim.qpos.copy(), sim.qvel.copy(), sim.qacc_warmstart.copy(), sim.ctrl.copy(),
                   np.stack([acts[a] for a in agents]))
            sim.step()
            post = {"qpos": sim.qpos.copy(), "qvel": sim.qvel.copy(), "sensordata": sim.sensordata.copy(),
                    "pairs": sorted(sim.contact_pairs()), "xipos": sim.xipos.copy()}
            out.append((pre, post))
        else:
            sim.step()
    return out
