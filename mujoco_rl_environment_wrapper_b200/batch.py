"""Batch: `num_envs` lock-stepped environments on one GPU behind the C-ABI (include/mjb.h).

Plays the role of `MjData` x num_envs (MuJoCo_Gym/mujoco_parent.py:127): all state lives in torch
CUDA tensors owned here (row-major, env-major, rows 16 B aligned); the library only gets raw device
pointers.  There is no CPU fallback: constructing a Batch without a CUDA device raises.
"""
import ctypes

import numpy as np
import torch

from . import _lib as L


class Batch:
    def __init__(self, model: "L.Model", spec: "L.EnvSpec", num_envs: int, device=None, keepalive=(), share=None, probe_quat=False):
        """`share`: another Batch whose tensors this handle steps as well (level variants, see set_subset);
        the two models must produce the same buffer layout."""
        self._lib = L.load()
        if not torch.cuda.is_available():
            raise RuntimeError("mujoco_rl_environment_wrapper_b200: no CUDA device — the step path is CUDA-only "
                               "(sm_100a); there is no CPU fallback")
        self.model, self.spec, self.num_envs = model, spec, int(num_envs)
        self._keep = keepalive
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        lay = L.Layout()
        L.check(self._lib.mjb_batch_layout(model._h, ctypes.byref(spec), self.num_envs, ctypes.byref(lay)), "batch layout")
        self.layout = lay
        if share is not None:
            same = all(getattr(lay, f) == getattr(share.layout, f) for f, _ in L.Layout._fields_)
            if not same or share.num_envs != self.num_envs or share.device != self.device:
                raise Exception("level variants must share one buffer layout (same sizes, sensors, agents and plugins)")
        A, N, dev = spec.n_agents, self.num_envs, self.device
        f32, i32, u8 = torch.float32, torch.int32, torch.uint8
        z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=dev)
        self.buf = share.buf if share is not None else {
            "qpos": z((N, lay.qpos_stride), f32), "qvel": z((N, lay.qvel_stride), f32),
            "ctrl": z((N, lay.ctrl_stride), f32), "warmstart": z((N, lay.qvel_stride), f32),
            "sensordata": z((N, lay.sensor_stride), f32), "probe": z((N, max(1, lay.probe_count), 4), f32),
            "actions": z((N, max(1, A), lay.act_stride), f32), "obs": z((N, max(1, A), lay.obs_stride), f32),
            "reward": z((N, max(1, A)), f32), "term": z((N, A + 1), u8), "trunc": z((N, A + 1), u8),
            "timestep": z((N,), i32), "store_i": z((N, max(1, A), lay.store_i32), i32),
            "store_f": z((N, max(1, A), lay.store_f32), f32), "ncon": z((N,), i32),
            "contact_geom": z((N, lay.maxcon, 2), i32), "contact_dist": z((N, lay.maxcon), f32), "niter": z((N,), i32), "nreset": z((N,), i32), "ncon_dropped": z((N,), i32),
        }
        if share is None and probe_quat and lay.probe_count > 0:
            q = z((N, lay.probe_count, 4), f32)
            q[:, :, 0] = 1.0
            self.buf["probe_quat"] = q
        B = L.Buffers()
        for k, v in self.buf.items():
            setattr(B, k, v.data_ptr())
        self._B = B
        self.stream = torch.cuda.current_stream(dev)
        h = ctypes.c_void_p()
        with torch.cuda.device(dev):
            L.check(self._lib.mjb_batch_create(model._h, ctypes.byref(spec), self.num_envs, dev.index or 0,
                                               ctypes.c_void_p(self.stream.cuda_stream), ctypes.byref(B), ctypes.byref(h)),
                    "batch create")
        self._h = h

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                self._lib.mjb_batch_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def __getattr__(self, k):
        buf = self.__dict__.get("buf")
        if buf is not None and k in buf:
            return buf[k]
        raise AttributeError(k)

    # ---- device-side entry points (asynchronous on self.stream)
    def reset(self, mask=None):
        p = None
        if mask is not None:
            self._mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
            p = ctypes.c_void_p(self._mask.data_ptr())
        L.check(self._lib.mjb_reset(self._h, p), "reset")

    def step(self):
        L.check(self._lib.mjb_step(self._h), "step")

    def set_subset(self, env_ids=None):
        """Restrict this handle's launches to the listed env indices (int32 CUDA tensor; None = all envs)."""
        if env_ids is None:
            self._subset = None
            L.check(self._lib.mjb_set_env_subset(self._h, None, 0), "env subset")
            return
        ids = env_ids.to(device=self.device, dtype=torch.int32).contiguous()
        count = int(ids.numel())
        if count == 0:
            # a zero-element tensor has data_ptr() == 0, and NULL means "all envs" to the C side: an empty level
            # must stay empty, so hand over a valid one-element dummy with count = 0
            ids = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._subset = ids
        L.check(self._lib.mjb_set_env_subset(self._h, ctypes.c_void_p(self._subset.data_ptr()), count), "env subset")

    def render(self, cam_ids, width=64, height=64, out=None):
        """u8 [num_envs, len(cam_ids), height, width, 3] images of the listed fixed cameras at the current qpos
        (rows bottom-up, like the reference's glReadPixels buffer).  Asynchronous on self.stream."""
        n = len(cam_ids)
        if out is None:
            out = torch.empty((self.num_envs, n, height, width, 3), dtype=torch.uint8, device=self.device)
        ids = (ctypes.c_int32 * n)(*cam_ids)
        L.check(self._lib.mjb_render(self._h, ids, n, int(width), int(height), ctypes.c_void_p(out.data_ptr())), "render")
        return out

    def physics(self, skip_frames=1):
        L.check(self._lib.mjb_physics(self._h, skip_frames), "physics")

    def forward(self):
        L.check(self._lib.mjb_forward(self._h), "forward")

    def sync(self):
        L.check(self._lib.mjb_sync(self._h), "sync")

    # ---- host-buffer step: numpy in / numpy out, copies inside
    def step_host(self, actions: np.ndarray, obs: np.ndarray, reward: np.ndarray, term: np.ndarray, trunc: np.ndarray):
        """One step through host arrays.  With page-locked arrays (host_arrays()) the kernel writes the results into
        them directly and the device tensors self.obs / reward / term / trunc keep their previous contents
        (include/mjb.h, mjb_step_host); the state tensors are always current."""
        L.check(self._lib.mjb_step_host(self._h, actions.ctypes.data, obs.ctypes.data, reward.ctypes.data,
                                        term.ctypes.data, trunc.ctypes.data), "step_host")

    def host_arrays(self, pinned=True):
        """(actions, obs, reward, term, trunc) host arrays for step_host.  Page-locked by default: the library
        then copies the actions straight from them and the kernel writes the results into them; pageable arrays work
        too (staged through pinned memory)."""
        lay, A, N = self.layout, self.spec.n_agents, self.num_envs
        z = lambda shape, dt: torch.zeros(shape, dtype=dt, pin_memory=pinned)
        f32, u8 = torch.float32, torch.uint8
        self._host_keep = [z((N, A, lay.act_stride), f32), z((N, A, lay.obs_stride), f32), z((N, A), f32),
                           z((N, A + 1), u8), z((N, A + 1), u8)]
        return tuple(t.numpy() for t in self._host_keep)

    @property
    def launch_count(self):
        return int(self._lib.mjb_launch_count(self._h))

    def set_timing(self, enable=True):
        L.check(self._lib.mjb_set_timing(self._h, 1 if enable else 0))

    def kernel_time_ms(self):
        t, n = ctypes.c_double(), ctypes.c_int64()
        L.check(self._lib.mjb_kernel_time_ms(self._h, ctypes.byref(t), ctypes.byref(n)))
        return t.value, n.value

    def geometry(self):
        g, w, s = ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int64()
        self._lib.mjb_batch_geometry(self._h, ctypes.byref(g), ctypes.byref(w), ctypes.byref(s))
        return {"grid": g.value, "warps_per_cta": w.value, "smem_bytes": s.value}
