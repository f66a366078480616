"""ctypes binding of include/mjb.h (libmjb.so).  No torch types cross this boundary: plain
pointers, sizes and POD structs only."""
import ctypes
import os
import struct

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# MJB_LIB selects a differently built copy of the same library (debug tooling: the phase-profile build of tools/)
LIB_PATH = os.environ.get("MJB_LIB") or os.path.join(_HERE, "libmjb.so")

MAX_AGENTS, MAX_PLUGINS, MAX_TARGETS, MAX_EXTRA_PROBES = 8, 4, 16, 48
SPEC_NO_PACK = 1   # mjb_env_spec.flags
OBJ_BODY, OBJ_JOINT, OBJ_GEOM, OBJ_SITE, OBJ_CAMERA, OBJ_ACTUATOR, OBJ_SENSOR = 1, 3, 5, 6, 7, 19, 20
DYN_LANGUAGE, DYN_PICKUP = 1, 2
REW_TAG_DISTANCE, REW_ANT = 1, 2
DONE_DISTANCE_LE = 1
STORE_I = {"utterance": 0, "has_utterance": 1, "current_target": 2, "inventory": 3, "has_xpos": 4, "draws": 5}
STORE_I_COUNT = 8
STORE_F = {"distance": 0, "xpos_before": 1}
STORE_F_COUNT = 4
JNT_FREE, JNT_SLIDE, JNT_HINGE = 0, 2, 3


class Dims(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in
                ("nq", "nv", "nu", "nbody", "njnt", "ngeom", "nsite", "nsensor", "nsensordata", "npair",
                 "integrator", "ncam")] + [("timestep", ctypes.c_double)]


class Plugin(ctypes.Structure):
    _fields_ = [("kind", ctypes.c_int32), ("act_lo", ctypes.c_int32), ("act_hi", ctypes.c_int32),
                ("n_obs", ctypes.c_int32), ("param", ctypes.c_float * 4)]


class EnvSpec(ctypes.Structure):
    _fields_ = [
        ("n_agents", ctypes.c_int32), ("free_joint", ctypes.c_int32), ("skip_frames", ctypes.c_int32),
        ("max_steps", ctypes.c_int32), ("n_phys_act", ctypes.c_int32), ("act_dim", ctypes.c_int32),
        ("obs_dim", ctypes.c_int32 * MAX_AGENTS), ("agent_body", ctypes.c_int32 * MAX_AGENTS),
        ("act_index", ctypes.POINTER(ctypes.c_int32)), ("obs_index", ctypes.POINTER(ctypes.c_int32)),
        ("obs_adr", ctypes.c_int32 * (MAX_AGENTS + 1)),
        ("n_dynamics", ctypes.c_int32), ("n_rewards", ctypes.c_int32), ("n_dones", ctypes.c_int32),
        ("dynamics", Plugin * MAX_PLUGINS), ("rewards", Plugin * MAX_PLUGINS), ("dones", Plugin * MAX_PLUGINS),
        ("n_targets", ctypes.c_int32),
        ("target_objtype", ctypes.c_int32 * MAX_TARGETS), ("target_objid", ctypes.c_int32 * MAX_TARGETS),
        ("seed", ctypes.c_uint64),
        ("solver_iterations", ctypes.c_int32), ("ls_iterations", ctypes.c_int32), ("flags", ctypes.c_int32), ("reset_noise", ctypes.c_float),
        ("n_extra_probes", ctypes.c_int32), ("extra_objtype", ctypes.c_int32 * MAX_EXTRA_PROBES), ("extra_objid", ctypes.c_int32 * MAX_EXTRA_PROBES),
    ]


class Layout(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in
                ("num_envs", "qpos_stride", "qvel_stride", "ctrl_stride", "sensor_stride", "act_stride",
                 "obs_stride", "probe_count", "maxcon", "store_i32", "store_f32")]


class Buffers(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in
                ("qpos", "qvel", "ctrl", "warmstart", "sensordata", "probe", "actions", "obs", "reward", "term",
                 "trunc", "timestep", "store_i", "store_f", "ncon", "contact_geom", "contact_dist", "niter", "nreset", "probe_quat", "ncon_dropped")]


_LIB = None


def load(build_if_missing=True):
    """Load libmjb.so; builds it in-tree with nvcc when missing or stale (CPU container only)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if build_if_missing and not os.environ.get("MJB_LIB"):
        from . import build as _build
        try:
            if _build.needs_build():
                _build.build()
        except Exception:
            if not os.path.exists(LIB_PATH):
                raise
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -m mujoco_rl_environment_wrapper_b200.build` "
                           "(there is no CPU fallback for the step path)")
    lib = ctypes.CDLL(LIB_PATH)
    vp, i32, i64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64
    lib.mjb_last_error.restype = ctypes.c_char_p
    lib.mjb_version.restype = ctypes.c_char_p
    lib.mjb_model_create.argtypes = [ctypes.c_char_p, ctypes.POINTER(vp)]
    lib.mjb_model_destroy.argtypes = [vp]
    lib.mjb_model_destroy.restype = None
    lib.mjb_model_dims.argtypes = [vp, ctypes.POINTER(Dims)]
    lib.mjb_model_blob.restype = vp
    lib.mjb_model_blob.argtypes = [vp, ctypes.POINTER(i64)]
    lib.mjb_name2id.argtypes = [vp, ctypes.c_int, ctypes.c_char_p]
    lib.mjb_id2name.restype = ctypes.c_char_p
    lib.mjb_id2name.argtypes = [vp, ctypes.c_int, ctypes.c_int]
    lib.mjb_batch_layout.argtypes = [vp, ctypes.POINTER(EnvSpec), i32, ctypes.POINTER(Layout)]
    lib.mjb_batch_create.argtypes = [vp, ctypes.POINTER(EnvSpec), i32, i32, vp, ctypes.POINTER(Buffers),
                                     ctypes.POINTER(vp)]
    lib.mjb_batch_destroy.argtypes = [vp]
    lib.mjb_batch_destroy.restype = None
    lib.mjb_reset.argtypes = [vp, vp]
    lib.mjb_step.argtypes = [vp]
    lib.mjb_physics.argtypes = [vp, i32]
    lib.mjb_forward.argtypes = [vp]
    lib.mjb_sync.argtypes = [vp]
    lib.mjb_step_host.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.mjb_launch_count.restype = i64
    lib.mjb_launch_count.argtypes = [vp]
    lib.mjb_set_timing.argtypes = [vp, i32]
    lib.mjb_kernel_time_ms.argtypes = [vp, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(i64)]
    lib.mjb_set_env_subset.argtypes = [vp, vp, ctypes.c_int32]
    lib.mjb_render.argtypes = [vp, ctypes.POINTER(ctypes.c_int32), ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, vp]
    lib.mjb_batch_geometry.argtypes = [vp, ctypes.POINTER(i32), ctypes.POINTER(i32), ctypes.POINTER(i64)]
    lib.mjb_phase_cycles.argtypes = [ctypes.POINTER(ctypes.c_uint64), i32]
    lib.mjb_draw_u32.restype = ctypes.c_uint32
    lib.mjb_draw_u32.argtypes = [ctypes.c_uint64, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32]
    _LIB = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().mjb_last_error().decode(errors="replace")
        raise Exception(f"{what}: {msg}" if what else msg)


def parse_blob(raw: bytes):
    """Packed model blob (include/mjb_blob.h) -> {field: numpy array} (copies)."""
    magic, nf, _, _tot = struct.unpack_from("8siiq", raw, 0)
    if not magic.startswith(b"MJBLOB1"):
        raise ValueError("bad model blob")
    out = {}
    for i in range(nf):
        name, dt, cnt, off = struct.unpack_from("32siiq", raw, 24 + i * 48)
        name = name.split(b"\0")[0].decode()
        out[name] = np.frombuffer(raw, dtype=np.int32 if dt == 0 else np.float64, count=cnt, offset=off).copy()
    return out


class Model:
    """Compiled MJCF model (host side). Plays the role of `MjModel` for name / size queries."""

    def __init__(self, xml_text: str):
        self._lib = load()
        h = ctypes.c_void_p()
        check(self._lib.mjb_model_create(xml_text.encode(), ctypes.byref(h)), "MJCF compile")
        self._h = h
        d = Dims()
        check(self._lib.mjb_model_dims(h, ctypes.byref(d)))
        self.dims = d
        n = ctypes.c_int64()
        p = self._lib.mjb_model_blob(h, ctypes.byref(n))
        self.blob = bytes((ctypes.c_char * n.value).from_address(p))
        self.fields = parse_blob(self.blob)
        for k in ("nq", "nv", "nu", "nbody", "njnt", "ngeom", "nsite", "nsensor", "nsensordata", "npair", "ncam"):
            setattr(self, k, getattr(d, k))
        self.timestep = d.timestep

    @classmethod
    def from_xml_path(cls, path):
        with open(path, "r") as f:
            return cls(f.read())

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                self._lib.mjb_model_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def name2id(self, objtype, name):
        return self._lib.mjb_name2id(self._h, objtype, name.encode())

    def id2name(self, objtype, idx):
        r = self._lib.mjb_id2name(self._h, objtype, idx)
        return None if r is None else r.decode()
