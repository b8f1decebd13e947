"""ctypes binding of the C ABI (include/deepmimic_b200.h).  Device buffers are torch CUDA tensors; torch is only
the allocator / stream plumbing here.  Raises if the CUDA library is missing -- there is no CPU fallback."""
import ctypes as C
import os

import numpy as np

_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_LIB_PATH = os.environ.get("DM_LIB", os.path.join(_REPO, "deepmimic_b200", "libdeepmimic_b200.so"))   # DM_LIB: profile build (tools/section_profile.py)
_lib = None


class DmDims(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("num_envs", "num_joints", "pose_dim", "num_dofs", "state_size", "goal_size", "action_size", "snapshot_size",
                                        "updates_per_action", "num_update_substeps")] + [("motion_duration", C.c_double), ("amp_obs_size", C.c_int)]


DM_STATE_OFFSET, DM_STATE_SCALE, DM_ACTION_OFFSET, DM_ACTION_SCALE, DM_ACTION_BOUND_MIN, DM_ACTION_BOUND_MAX, DM_STATE_NORM_GROUPS = range(7)

EXPORTS = ["dm_create", "dm_load_host", "dm_plan_launch", "dm_get_model_info", "dm_get_link_table", "dm_destroy", "dm_last_error", "dm_get_dims", "dm_get_static", "dm_get_scene_name", "dm_stream", "dm_sync", "dm_set_mode", "dm_set_sample_count", "dm_get_time_limits", "dm_reset", "dm_set_action",
           "dm_update", "dm_record_state", "dm_record_goal", "dm_goal_host", "dm_reset_clips", "dm_record_amp_obs_expert_clips", "dm_get_clip_table", "dm_get_task_state", "dm_set_task_state", "dm_get_task_params", "dm_calc_reward", "dm_calc_reward_imitate", "dm_record_amp_obs_agent", "dm_record_amp_obs_expert", "dm_amp_obs_host", "dm_observe", "dm_get_flags", "dm_step_host", "dm_step_host_reset", "dm_set_time_limits", "dm_exchange_create", "dm_exchange_connect", "dm_exchange_publish", "dm_exchange_acquire", "dm_exchange_release", "dm_exchange_status", "dm_exchange_destroy", "dm_set_timing", "dm_step_host_timing", "dm_get_snapshot",
           "dm_set_snapshot", "dm_get_counters", "dm_debug_enable", "dm_get_debug", "dm_mlp_create", "dm_mlp_forward", "dm_mlp_launches", "dm_mlp_destroy"]


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise RuntimeError("deepmimic_b200: %s is missing -- run `python -c 'import __graft_entry__ as g; g.build()'`. "
                               "There is no CPU fallback." % _LIB_PATH)
        L = C.CDLL(_LIB_PATH)
        vp, dp, fp, ip = C.c_void_p, C.POINTER(C.c_double), C.c_void_p, C.c_void_p
        L.dm_create.restype = vp
        L.dm_create.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.c_char_p), C.c_int, C.c_int, C.c_uint64, C.c_uint64]
        L.dm_destroy.argtypes = [vp]
        L.dm_load_host.restype = vp
        L.dm_load_host.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.c_char_p)]
        L.dm_get_model_info.argtypes = [vp, C.c_int, C.POINTER(C.c_int)]
        L.dm_plan_launch.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int)]
        L.dm_get_link_table.argtypes = [vp, dp]
        L.dm_last_error.restype = C.c_char_p
        L.dm_get_dims.argtypes = [vp, C.POINTER(DmDims)]
        L.dm_get_static.argtypes = [vp, C.c_int, dp]
        L.dm_get_scene_name.argtypes = [vp, C.c_char_p, C.c_int]
        L.dm_stream.restype = vp
        L.dm_stream.argtypes = [vp]
        L.dm_sync.argtypes = [vp]
        L.dm_set_mode.argtypes = [vp, C.c_int]
        L.dm_set_sample_count.argtypes = [vp, C.c_longlong]
        L.dm_get_time_limits.argtypes = [vp, dp]
        L.dm_reset.argtypes = [vp, C.c_int, dp, dp, dp]
        L.dm_set_action.argtypes = [vp, fp]
        L.dm_update.argtypes = [vp, C.c_double, C.c_int]
        L.dm_record_state.argtypes = [vp, fp]
        L.dm_record_goal.argtypes = [vp, fp]
        L.dm_calc_reward.argtypes = [vp, fp]
        L.dm_calc_reward_imitate.argtypes = [vp, fp]
        L.dm_goal_host.argtypes = [vp, fp]
        L.dm_reset_clips.argtypes = [vp, C.c_int, C.POINTER(C.c_int), dp, dp, dp]
        L.dm_record_amp_obs_expert_clips.argtypes = [vp, C.POINTER(C.c_int), dp, fp]
        L.dm_get_clip_table.argtypes = [vp, C.POINTER(C.c_int), dp, dp]
        L.dm_get_task_state.argtypes = [vp, C.c_int, dp]
        L.dm_set_task_state.argtypes = [vp, C.c_int, dp]
        L.dm_get_task_params.argtypes = [vp, dp, C.POINTER(C.c_uint64)]
        L.dm_record_amp_obs_agent.argtypes = [vp, fp]
        L.dm_record_amp_obs_expert.argtypes = [vp, dp, fp]
        L.dm_amp_obs_host.argtypes = [vp, C.c_int, dp, fp]
        L.dm_observe.argtypes = [vp, fp, fp]
        L.dm_get_flags.argtypes = [vp, ip]
        L.dm_step_host.argtypes = [vp, fp, C.c_double, C.c_int, fp, fp, ip]
        L.dm_step_host_reset.argtypes = [vp, fp, C.c_double, C.c_int, fp, fp, ip, C.c_int]
        L.dm_set_time_limits.argtypes = [vp, C.c_double, C.c_double]
        L.dm_exchange_create.argtypes = [vp, C.c_int, C.c_int, C.c_void_p]
        L.dm_exchange_connect.argtypes = [vp, C.c_void_p]
        L.dm_exchange_publish.argtypes = [vp, C.c_longlong]
        L.dm_exchange_acquire.argtypes = [vp, C.c_longlong, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]
        L.dm_exchange_release.argtypes = [vp, C.c_longlong]
        L.dm_exchange_status.argtypes = [vp, C.POINTER(C.c_int)]
        L.dm_exchange_destroy.argtypes = [vp]
        L.dm_set_timing.argtypes = [vp, C.c_int]
        L.dm_step_host_timing.argtypes = [vp, dp]
        L.dm_get_snapshot.argtypes = [vp, C.c_int, dp]
        L.dm_set_snapshot.argtypes = [vp, C.c_int, dp]
        L.dm_get_counters.argtypes = [vp, C.POINTER(C.c_int64)]
        L.dm_debug_enable.argtypes = [vp, C.c_int]
        L.dm_get_debug.argtypes = [vp, C.c_int, C.c_void_p]
        fpp = C.POINTER(C.c_float)
        L.dm_mlp_create.restype = vp
        L.dm_mlp_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, fpp, fpp, fpp, fpp, fpp, fpp, fpp, fpp, C.c_float, fpp, fpp, C.c_int]
        L.dm_mlp_forward.argtypes = [vp, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.dm_mlp_launches.restype = C.c_longlong
        L.dm_mlp_launches.argtypes = [vp]
        L.dm_mlp_destroy.argtypes = [vp]
        _lib = L
    return _lib


def _dptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_double)) if a is not None else None


class _Handle:
    """What a device handle (dm_create) and a host-only handle (dm_load_host) share: the host model's tables, the launch plan, close()."""
    h = None

    def _open(self, create, args, asset_root, *extra):
        enc = [a.encode() for a in args]
        h = create(asset_root.encode(), len(enc), (C.c_char_p * len(enc))(*enc), *extra)
        if not h:
            raise RuntimeError("%s failed: %s" % (create.__name__, lib().dm_last_error().decode()))
        self.h = C.c_void_p(h)
        self.dims = DmDims()
        self._chk(lib().dm_get_dims(self.h, C.byref(self.dims)))

    def _chk(self, rc):
        if rc != 0:
            raise RuntimeError("deepmimic_b200: %s" % lib().dm_last_error().decode())

    def close(self):
        if self.h:
            lib().dm_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def static(self, kind):
        n = self.dims.state_size if kind in (DM_STATE_OFFSET, DM_STATE_SCALE, DM_STATE_NORM_GROUPS) else self.dims.action_size
        out = np.zeros(n, dtype=np.float64)
        self._chk(lib().dm_get_static(self.h, kind, _dptr(out)))
        return out

    def plan_launch(self, num_envs, smem_bytes_per_block=232448, num_sms=148):
        """dm_plan_launch: launch plan of the step kernel on a device with that much opt-in shared memory per block and that many SMs (B200 defaults)"""
        out = (C.c_int * 9)()
        self._chk(lib().dm_plan_launch(self.h, int(num_envs), int(smem_bytes_per_block), int(num_sms), out))
        keys = ("tile_width", "envs_per_block", "blocks", "smem_bytes", "max_rows", "env_floats", "hot_floats", "y_offset", "padded_envs")
        return dict(zip(keys, [int(v) for v in out]))

    def task_params(self):
        out = np.zeros(48, dtype=np.float64)     # [0:16] dm_task.cuh constants, [16:48] dm_task_ext.cuh constants
        key = (C.c_uint64 * 2)()
        self._chk(lib().dm_get_task_params(self.h, _dptr(out), key))
        return out, int(key[0]), int(key[1])

    def clip_table(self):
        n = C.c_int(0)
        self._chk(lib().dm_get_clip_table(self.h, C.byref(n), None, None))
        dur, cdf = np.zeros(n.value), np.zeros(n.value)
        self._chk(lib().dm_get_clip_table(self.h, C.byref(n), _dptr(dur), _dptr(cdf)))
        return dur, cdf

    def set_sample_count(self, count):
        self._chk(lib().dm_set_sample_count(self.h, int(count)))

    def time_limits(self):
        out = np.zeros(3, dtype=np.float64)
        self._chk(lib().dm_get_time_limits(self.h, _dptr(out)))
        return out


class BatchedCore(_Handle):
    """Thin object wrapper over a dm_handle."""

    def __init__(self, args, num_envs, asset_root, device=0, seed=0, global_env_offset=0):
        self._open(lib().dm_create, args, asset_root, num_envs, device, seed, global_env_offset)
        self.num_envs = self.dims.num_envs

    def scene_name(self):
        buf = C.create_string_buffer(64)
        self._chk(lib().dm_get_scene_name(self.h, buf, 64))
        return buf.value.decode()

    def reset(self, force_all=True, kin_time=None, max_time=None, rot_theta=None, clip=None):
        f = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float64)
        kt, mt, th = f(kin_time), f(max_time), f(rot_theta)
        if clip is None:
            self._chk(lib().dm_reset(self.h, 1 if force_all else 0, _dptr(kt), _dptr(mt), _dptr(th)))
        else:   # task scenes with a clip dataset: the controller's clip draw injected
            c = np.ascontiguousarray(clip, dtype=np.int32)
            self._chk(lib().dm_reset_clips(self.h, 1 if force_all else 0, c.ctypes.data_as(C.POINTER(C.c_int)), _dptr(kt), _dptr(mt), _dptr(th)))

    def set_action(self, actions):  # torch float32 cuda tensor [N, A]
        self._chk(lib().dm_set_action(self.h, C.c_void_p(actions.data_ptr())))

    def update(self, dt, n_updates=1):
        self._chk(lib().dm_update(self.h, dt, n_updates))

    def observe(self, state=None, reward=None):
        self._chk(lib().dm_observe(self.h, C.c_void_p(state.data_ptr()) if state is not None else None,
                                   C.c_void_p(reward.data_ptr()) if reward is not None else None))

    def reward_imitate(self, out):  # torch float32 cuda tensor [N]: CalcRewardImitate also in the task scenes (active clip of the dataset)
        self._chk(lib().dm_calc_reward_imitate(self.h, C.c_void_p(out.data_ptr())))

    def record_goal(self, out):  # torch float32 cuda tensor [N, goal_size]; task scenes only
        self._chk(lib().dm_record_goal(self.h, C.c_void_p(out.data_ptr())))

    def goal_host(self):
        out = np.zeros((self.num_envs, self.dims.goal_size), dtype=np.float32)
        self._chk(lib().dm_goal_host(self.h, C.c_void_p(out.ctypes.data)))
        return out

    def task_state(self, env):
        out = np.zeros(24, dtype=np.float64)     # dm_task.cuh block (16) | dm_task_ext.cuh block (8)
        self._chk(lib().dm_get_task_state(self.h, env, _dptr(out)))
        return out

    def set_task_state(self, env, block):
        b = np.ascontiguousarray(block, dtype=np.float64)
        self._chk(lib().dm_set_task_state(self.h, env, _dptr(b)))

    def amp_obs_agent(self, out):  # torch float32 cuda tensor [N, amp_obs_size]
        self._chk(lib().dm_record_amp_obs_agent(self.h, C.c_void_p(out.data_ptr())))

    def amp_obs_expert(self, out, kin_time=None, clip=None):
        kt = None if kin_time is None else np.ascontiguousarray(kin_time, dtype=np.float64)
        if clip is None:
            self._chk(lib().dm_record_amp_obs_expert(self.h, _dptr(kt), C.c_void_p(out.data_ptr())))
        else:
            c = np.ascontiguousarray(clip, dtype=np.int32)
            self._chk(lib().dm_record_amp_obs_expert_clips(self.h, c.ctypes.data_as(C.POINTER(C.c_int)), _dptr(kt), C.c_void_p(out.data_ptr())))

    def flags(self, out):  # torch int32 cuda tensor [N, 4]
        self._chk(lib().dm_get_flags(self.h, C.c_void_p(out.data_ptr())))

    def sync(self):
        self._chk(lib().dm_sync(self.h))

    def set_mode(self, mode):
        self._chk(lib().dm_set_mode(self.h, mode))

    def step_host(self, actions, dt, n_updates, state, reward, flags, reset_done=False):  # numpy host arrays
        p = lambda a: None if a is None else C.c_void_p(a.ctypes.data)
        self._chk(lib().dm_step_host_reset(self.h, p(actions), dt, n_updates, p(state), p(reward), p(flags), 1 if reset_done else 0))

    def set_episode_limit(self, seconds_min, seconds_max=None):
        self._chk(lib().dm_set_time_limits(self.h, float(seconds_min), float(seconds_min if seconds_max is None else seconds_max)))

    # ---- multi-GPU exchange over NVLink peer memory (dm_exchange_*)
    def exchange_create(self, rank, world):
        buf = C.create_string_buffer(64)
        self._chk(lib().dm_exchange_create(self.h, rank, world, buf))
        return bytes(buf.raw)

    def exchange_connect(self, handles):   # world x 64 bytes, rank order
        blob = b"".join(handles)
        self._chk(lib().dm_exchange_connect(self.h, C.c_char_p(blob)))

    def exchange_publish(self, step):
        self._chk(lib().dm_exchange_publish(self.h, int(step)))

    def exchange_acquire(self, step):
        o, r, d = C.c_void_p(), C.c_void_p(), C.c_void_p()
        self._chk(lib().dm_exchange_acquire(self.h, int(step), C.byref(o), C.byref(r), C.byref(d)))
        return o.value, r.value, d.value

    def exchange_release(self, step):
        self._chk(lib().dm_exchange_release(self.h, int(step)))

    def exchange_status(self):
        s = C.c_int(0)
        self._chk(lib().dm_exchange_status(self.h, C.byref(s)))
        return s.value

    def set_timing(self, on=True):
        self._chk(lib().dm_set_timing(self.h, 1 if on else 0))

    def step_host_timing(self):
        """last dm_step_host: dict of device ms per phase and host wall ms (enqueue / wait / staging copies)"""
        o = np.zeros(8, dtype=np.float64)
        self._chk(lib().dm_step_host_timing(self.h, _dptr(o)))
        return dict(h2d_set_action_ms=o[0], update_ms=o[1], observe_flags_ms=o[2], d2h_ms=o[3], host_enqueue_ms=o[4], host_wait_ms=o[5], host_copy_ms=o[6])

    def get_snapshot(self, env):
        out = np.zeros(self.dims.snapshot_size, dtype=np.float64)
        self._chk(lib().dm_get_snapshot(self.h, env, _dptr(out)))
        return out

    def set_snapshot(self, env, snap):
        s = np.ascontiguousarray(snap, dtype=np.float64)
        self._chk(lib().dm_set_snapshot(self.h, env, _dptr(s)))

    def counters(self):
        out = (C.c_int64 * 2)()
        self._chk(lib().dm_get_counters(self.h, out))
        return int(out[0]), int(out[1])

    def debug_enable(self, on=True):
        self._chk(lib().dm_debug_enable(self.h, 1 if on else 0))

    def get_debug(self, env):
        out = np.zeros(8 * 96 + 2048, dtype=np.float32)
        self._chk(lib().dm_get_debug(self.h, env, C.c_void_p(out.ctypes.data)))
        return out

    def stream(self):
        return lib().dm_stream(self.h)


class HostModel(_Handle):
    """dm_load_host handle: the host loaders and the flat model, no device (used by the CPU tests and by tools)."""
    INFO = dict(parents=0, joint_types=1, dof_offsets=2, pose_offsets=3, fall_bodies=4, end_effectors=5)

    def __init__(self, args, asset_root):
        self._open(lib().dm_load_host, args, asset_root)

    def info(self, name):
        out = (C.c_int * self.dims.num_joints)()
        self._chk(lib().dm_get_model_info(self.h, self.INFO[name], out))
        return np.array(out[:], dtype=np.int64)

    def link_table(self):
        """[num_joints, 24]: mass, inertiaB[3], inertiaD[3], dvec[3], evec[3], zrot xyzw, axis[3], half extents[3], breaking threshold"""
        out = np.zeros((self.dims.num_joints, 24), dtype=np.float64)
        self._chk(lib().dm_get_link_table(self.h, _dptr(out)))
        return out

    def layout(self):
        out = (C.c_int * 6)()
        self._chk(lib().dm_get_model_info(self.h, 6, out))
        return dict(zip(("links", "dofs", "chain_stride", "tree_depth", "frames", "loop"), out[:]))


class TensorCoreMLP:
    """dm_mlp_* handle: the actor network (normalise -> 2 hidden ReLU layers -> linear -> un-normalise) on the tcgen05 tensor cores.
    weights: the reference's dense kernels, [inputs x units] float arrays (deepmimic_b200.tf_checkpoint.load_actor / the fixture files)."""

    def __init__(self, w0, b0, w1, b1, w2, b2, in_mean=None, in_std=None, in_clip=float("inf"), out_mean=None, out_std=None, max_rows=4096, device=0):
        L = lib()
        f = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float32)
        w0, b0, w1, b1, w2, b2, in_mean, in_std, out_mean, out_std = (f(x) for x in (w0, b0, w1, b1, w2, b2, in_mean, in_std, out_mean, out_std))
        self.in_dim, self.h0 = w0.shape
        self.h1, self.out_dim = w2.shape
        assert w1.shape == (self.h0, self.h1) and b0.shape == (self.h0,) and b1.shape == (self.h1,) and b2.shape == (self.out_dim,)
        p = lambda a: None if a is None else a.ctypes.data_as(C.POINTER(C.c_float))
        clip = 0.0 if not np.isfinite(in_clip) else float(in_clip)
        self.h = L.dm_mlp_create(device, self.in_dim, self.h0, self.h1, self.out_dim, p(w0), p(b0), p(w1), p(b1), p(w2), p(b2), p(in_mean), p(in_std), clip, p(out_mean), p(out_std), max_rows)
        if not self.h:
            raise RuntimeError("dm_mlp_create failed: %s" % L.dm_last_error().decode())
        self.h = C.c_void_p(self.h)
        self.max_rows = max_rows

    def forward(self, obs, actions, noise=None, stream=None):
        """obs [rows, in_dim], actions [rows, out_dim] (written), noise [rows, out_dim] or None: contiguous float32 CUDA tensors; stream: cudaStream_t handle (int) or None"""
        rows = obs.shape[0]
        rc = lib().dm_mlp_forward(self.h, C.c_void_p(obs.data_ptr()), C.c_void_p(noise.data_ptr()) if noise is not None else None, C.c_void_p(actions.data_ptr()), rows,
                                  C.c_void_p(stream) if stream else None)
        if rc != 0:
            raise RuntimeError("dm_mlp_forward: %s" % lib().dm_last_error().decode())
        return actions

    def launches(self):
        return int(lib().dm_mlp_launches(self.h))

    def close(self):
        if self.h:
            lib().dm_mlp_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
