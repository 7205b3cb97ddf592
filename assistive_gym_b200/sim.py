"""BatchSim — numpy-facing wrapper of the C ABI (include/agphys.h) for N lock-step envs.

This is the object the `pybullet`-shaped shim and the env classes talk to.  All arrays are
env-major (`[N, k, c]`); the library transposes to its SoA device layout.  The CUDA library is
mandatory: construction raises if it cannot be loaded or no CUDA device is present.
"""
import ctypes as C

import numpy as np

from . import capi


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _f32(a, shape=None):
    if a is None:
        return None
    a = np.asarray(a, dtype=np.float32)
    if shape is not None:
        a = np.broadcast_to(a, shape)
    return np.ascontiguousarray(a)


def _i32(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.int32)


class BatchSim:
    def __init__(self, scene, cfg=None, n_envs=1, device=0, _lib=None):
        self.lib = _lib if _lib is not None else capi.load_library()
        self.scene = scene
        self.cfg = cfg or capi.default_config()
        self.n = int(n_envs)
        self._desc = scene.as_ctypes()
        self.h = self.lib.ag_create(C.byref(self._desc), C.byref(self.cfg), self.n, int(device))
        if not self.h:
            raise RuntimeError('ag_create failed: %s' % self.lib.ag_last_error().decode())
        self.contact_dtype = capi.CONTACT_DTYPE
        for b in range(scene.n_bodies):
            self.set_base_pose(b, scene['base_pos0'][b], scene['base_quat0'][b])
        self.forward_kinematics()

    def _ck(self, rc):
        if rc != 0:
            raise RuntimeError(self.lib.ag_last_error().decode())

    # ---- the fused env steps (one call: action -> obs [n, obs_dim], reward [n], done [n], info [n, 4])
    def _step_host(self, fn, obs_dim, *action):
        """fn(sim, [action [n, 7],] obs, reward, done, info) on host arrays; returns (obs, reward, done, info)"""
        out = (np.empty((self.n, obs_dim), dtype=np.float32), np.empty(self.n, dtype=np.float32), np.empty(self.n, dtype=np.float32),
               np.empty((self.n, 4), dtype=np.float32))
        self._ck(fn(self.h, *[_p(_f32(a, (self.n, 7))) for a in action], *[_p(o) for o in out]))
        return out

    def _step_dev(self, fn, *ptrs):
        """device pointers (ints) to action [n, 7], obs, reward, done, info; asynchronous on the sim's stream"""
        self._ck(fn(self.h, *[C.c_void_p(p) for p in ptrs]))

    def close(self):
        if getattr(self, 'h', None):
            self.lib.ag_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- setters
    def set_base_pose(self, body, pos=None, quat=None, mask=None):
        pos, quat = _f32(pos, (self.n, 3)), _f32(quat, (self.n, 4))
        self._ck(self.lib.ag_set_base_pose(self.h, body, _p(pos), _p(quat), _p(_i32(mask))))

    def set_base_velocity(self, body, lin=None, ang=None, mask=None):
        lin, ang = _f32(lin, (self.n, 3)), _f32(ang, (self.n, 3))
        self._ck(self.lib.ag_set_base_velocity(self.h, body, _p(lin), _p(ang), _p(_i32(mask))))

    def set_joint_state(self, links, q=None, qd=None, mask=None):
        links = _i32(links)
        q, qd = _f32(q, (self.n, len(links))), _f32(qd, (self.n, len(links)))
        self._ck(self.lib.ag_set_joint_state(self.h, len(links), _p(links), _p(q), _p(qd), _p(_i32(mask))))

    def set_link_friction(self, link, mu, mask=None):
        mu = _f32(mu, (self.n,))
        self._ck(self.lib.ag_set_link_friction(self.h, int(link), _p(mu), _p(_i32(mask))))

    def set_body_active(self, body, active):
        m = _i32(np.broadcast_to(np.asarray(active, dtype=np.int32), (self.n,)))
        self._ck(self.lib.ag_set_body_active(self.h, body, _p(m)))

    def set_motor(self, links, mode, target=None, kp=None, kd=None, max_force=None):
        links = _i32(links)
        n = len(links)
        target = _f32(target, (self.n, n))
        kp = _f32(kp, (n,)) if kp is not None else None
        kd = _f32(kd if kd is not None else 1.0, (n,))
        mf = _f32(max_force, (n,)) if max_force is not None else None
        self._ck(self.lib.ag_set_motor_host(self.h, n, _p(links), int(mode), _p(target), _p(kp), _p(kd), _p(mf)))

    def set_motor_force_scale(self, links, scale):
        links = _i32(links)
        self._ck(self.lib.ag_set_motor_force_scale(self.h, len(links), _p(links), _p(_f32(scale, (self.n, len(links))))))

    def set_motor_targets(self, links, target):
        links = _i32(links)
        t = _f32(target, (self.n, len(links)))
        self._ck(self.lib.ag_set_motor_targets_host(self.h, len(links), _p(links), _p(t)))

    def set_body_gravity(self, body, g):
        gg = (C.c_double * 3)(*[float(a) for a in g])
        self._ck(self.lib.ag_set_body_gravity(self.h, int(body), gg))

    def get_link_aabb(self, links):
        links = _i32(links)
        mn = np.zeros((self.n, len(links), 3), dtype=np.float32)
        mx = np.zeros_like(mn)
        self._ck(self.lib.ag_get_link_aabb(self.h, len(links), _p(links), _p(mn), _p(mx)))
        return mn, mx

    def forward_kinematics(self):
        self._ck(self.lib.ag_forward_kinematics(self.h))

    def step(self, n_steps=1):
        self._ck(self.lib.ag_step(self.h, int(n_steps)))

    # ---- getters
    def get_joint_states(self, links):
        links = _i32(links)
        n = len(links)
        q, qd, tau = (np.zeros((self.n, n), dtype=np.float32) for _ in range(3))
        self._ck(self.lib.ag_get_joint_states(self.h, n, _p(links), _p(q), _p(qd), _p(tau)))
        return q, qd, tau

    def get_link_states(self, links):
        links = _i32(links)
        n = len(links)
        pos, cpos, lv, av = (np.zeros((self.n, n, 3), dtype=np.float32) for _ in range(4))
        quat, cquat = (np.zeros((self.n, n, 4), dtype=np.float32) for _ in range(2))
        self._ck(self.lib.ag_get_link_states(self.h, n, _p(links), _p(pos), _p(quat), _p(cpos), _p(cquat), _p(lv), _p(av)))
        return dict(pos=pos, quat=quat, com_pos=cpos, com_quat=cquat, lin_vel=lv, ang_vel=av)

    def get_contacts(self, body_a, body_b=-2, link_a=-2, link_b=-2, max_pts=64):
        out = np.zeros((self.n, max_pts), dtype=self.contact_dtype)
        cnt = np.zeros(self.n, dtype=np.int32)
        self._ck(self.lib.ag_get_contacts(self.h, body_a, body_b, link_a, link_b, max_pts, _p(out), _p(cnt)))
        return out, cnt

    def contact_force_sum(self, body_a, body_b=-2, link_a=-2, link_b=-2):
        out = np.zeros(self.n, dtype=np.float32)
        self._ck(self.lib.ag_contact_force_sum(self.h, body_a, body_b, link_a, link_b, _p(out)))
        return out

    def closest_points(self, body_a, body_b, distance, max_pts=64):
        out = np.zeros((self.n, max_pts), dtype=self.contact_dtype)
        cnt = np.zeros(self.n, dtype=np.int32)
        self._ck(self.lib.ag_closest_points(self.h, body_a, body_b, float(distance), max_pts, _p(out), _p(cnt)))
        return out, cnt

    def state_get(self):
        sz = self.lib.ag_state_size(self.h)
        out = np.zeros((self.n, sz), dtype=np.float32)
        self._ck(self.lib.ag_state_get(self.h, _p(out)))
        return out

    def state_set(self, st):
        st = _f32(st)
        self._ck(self.lib.ag_state_set(self.h, _p(st)))

    def kernel_launches(self):
        return int(self.lib.ag_kernel_launches(self.h))

    def overflow_count(self):
        return int(self.lib.ag_overflow_count(self.h))

    def solver_stats(self):
        c, it = np.zeros(self.n, dtype=np.int32), np.zeros(self.n, dtype=np.int32)
        self._ck(self.lib.ag_get_solver_stats(self.h, _p(c), _p(it)))
        return c, it

    def pgs_cycles(self):
        c = np.zeros(self.n, dtype=np.int32)
        self._ck(self.lib.ag_get_pgs_cycles(self.h, _p(c)))
        return c

    def pgs_trips(self):
        """(records consumed by the env's warp, floats of the env's row stream) of the last PGS launch."""
        t = np.zeros(self.n, dtype=np.int32)
        f = np.zeros(self.n, dtype=np.int32)
        self._ck(self.lib.ag_get_pgs_trips(self.h, _p(t), _p(f)))
        return t, f

    def profile_enable(self, on=True):
        self._ck(self.lib.ag_profile_enable(self.h, int(bool(on))))

    def profile_get(self):
        """{kernel name: (total ms, launches)} since the last call."""
        mx, stride = 32, 48
        names = C.create_string_buffer(mx * stride)
        ms = np.zeros(mx, dtype=np.float32)
        cnt = np.zeros(mx, dtype=np.int32)
        n = self.lib.ag_profile_get(self.h, mx, names, stride, _p(ms), _p(cnt))
        out = {}
        for i in range(max(n, 0)):
            nm = names.raw[i * stride:(i + 1) * stride].split(b'\0')[0].decode()
            out[nm] = (float(ms[i]), int(cnt[i]))
        return out

    def stream_ptr(self):
        return int(self.lib.ag_stream(self.h) or 0)

    # ---- fused feeding path
    def feeding_init(self, params, gender_is_male):
        self._feed_params = params
        g = _i32(np.broadcast_to(np.asarray(gender_is_male, dtype=np.int32), (self.n,)))
        self._ck(self.lib.ag_feeding_init(self.h, C.byref(params), _p(g)))

    def set_hard_limits(self, links, on=True):
        links = _i32(links)
        self._ck(self.lib.ag_set_hard_limits(self.h, len(links), _p(links), int(bool(on))))

    def feeding_set_tremor(self, on, rest, amplitude):
        o = _i32(np.broadcast_to(np.asarray(on, dtype=np.int32), (self.n,)))
        self._ck(self.lib.ag_feeding_set_tremor(self.h, _p(o), _p(_f32(rest, (self.n, 4))), _p(_f32(amplitude, (self.n, 4)))))

    def ik_solve(self, joint_links, ee_link, target_pos, target_quat, max_restarts=20, iters=120, threshold=0.01, seed=1, mask=None):
        """Batched DLS IK with random restarts on the device (robot.py:84-121); returns q [n, n_joints], err [n]."""
        jl = _i32(joint_links)
        tp = _f32(target_pos, (self.n, 3)); tq = _f32(np.broadcast_to(np.asarray(target_quat, dtype=np.float32), (self.n, 4)))
        q = np.zeros((self.n, len(jl)), dtype=np.float32); err = np.zeros(self.n, dtype=np.float32)
        self._ck(self.lib.ag_ik_solve(self.h, len(jl), _p(jl), int(ee_link), _p(tp), _p(tq), int(max_restarts), int(iters), float(threshold),
                                      int(seed), _p(_i32(mask)), _p(q), _p(err)))
        return q, err

    # ---- fused bed-bathing path
    def bathing_init(self, params, gender_is_male, targets_world, targets_valid):
        g = _i32(np.broadcast_to(np.asarray(gender_is_male, dtype=np.int32), (self.n,)))
        T = int(params.n_targets_max)
        tw = _f32(targets_world, (self.n, T, 3)); tv = _i32(np.ascontiguousarray(targets_valid, dtype=np.int32).reshape(self.n, T))
        self._ck(self.lib.ag_bathing_init(self.h, C.byref(params), _p(g), _p(tw), _p(tv)))

    def bathing_step_host(self, action):
        return self._step_host(self.lib.ag_bathing_step_host, 24, action)

    def bathing_step_dev(self, action_ptr, obs_ptr, reward_ptr, done_ptr, info_ptr):
        self._step_dev(self.lib.ag_bathing_step_dev, action_ptr, obs_ptr, reward_ptr, done_ptr, info_ptr)

    # ---- cloth (ag_cloth_*; node arrays in the PUBLIC node order of the ClothModel)
    def cloth_init(self, model, col_links, col_static, anchor_nodes, anchor_local, gravity=(0, 0, -9.81), max_contacts=1024):
        self.cloth_model = model
        self._cloth_desc = capi.make_cloth_desc(model, self.scene, col_links, col_static, anchor_nodes, anchor_local, gravity, max_contacts)
        self._ck(self.lib.ag_cloth_init(self.h, C.byref(self._cloth_desc)))

    def cloth_set_state(self, x=None, v=None, mask=None):
        m = self.cloth_model
        xi = None if x is None else _f32(m.to_internal(np.asarray(x)), (self.n, m.n_nodes, 3))
        vi = None if v is None else _f32(m.to_internal(np.asarray(v)), (self.n, m.n_nodes, 3))
        mk = None if mask is None else _i32(mask)
        self._ck(self.lib.ag_cloth_set_state(self.h, _p(xi), _p(vi), _p(mk)))

    def cloth_get_state(self):
        m = self.cloth_model
        x = np.empty((self.n, m.n_nodes, 3), dtype=np.float32)
        v = np.empty_like(x)
        self._ck(self.lib.ag_cloth_get_state(self.h, _p(x), _p(v)))
        return m.to_public(x), m.to_public(v)

    def cloth_set_anchor(self, pos, mask=None):
        mk = None if mask is None else _i32(mask)
        self._ck(self.lib.ag_cloth_set_anchor(self.h, _p(_f32(pos, (self.n, 3))), _p(mk)))

    def cloth_anchor_follow(self, link):
        self._ck(self.lib.ag_cloth_anchor_follow(self.h, int(link)))

    def cloth_set_gravity(self, g):
        gg = (C.c_double * 3)(*[float(a) for a in g])
        self._ck(self.lib.ag_cloth_set_gravity(self.h, gg))

    def cloth_get_contacts(self, max_pts=1024):
        cnt = np.zeros(self.n, dtype=np.int32)
        node = np.zeros((self.n, max_pts), dtype=np.int32)
        link = np.zeros((self.n, max_pts), dtype=np.int32)
        pos = np.zeros((self.n, max_pts, 3), dtype=np.float32)
        force = np.zeros((self.n, max_pts, 3), dtype=np.float32)
        self._ck(self.lib.ag_cloth_get_contacts(self.h, max_pts, _p(cnt), _p(node), _p(pos), _p(force), _p(link)))
        return cnt, self.cloth_model.order[node], pos, force, link

    # ---- fused scratch-itch path
    def scratch_init(self, params, gender_is_male, limb_link, target_local):
        self._scratch_params = params
        self._ck(self.lib.ag_scratch_init(self.h, C.byref(params), _p(_i32(gender_is_male)), _p(_i32(limb_link)), _p(_f32(target_local, (self.n, 3)))))

    def scratch_step_host(self, action):
        return self._step_host(self.lib.ag_scratch_step_host, 30, action)

    def scratch_step_dev(self, action_ptr, obs_ptr, reward_ptr, done_ptr, info_ptr):
        self._step_dev(self.lib.ag_scratch_step_dev, action_ptr, obs_ptr, reward_ptr, done_ptr, info_ptr)

    # ---- camera images (ag_render)
    def render(self, eye, target, fov=60.0, width=480, height=270, env_ids=(0,), up=(0, 0, 1), near=0.01, far=100.0,
               light_dir=(0, -3, 1), ambient=0.8, diffuse=0.3):
        cam = capi.AgCamera(eye=(C.c_float * 3)(*eye), target=(C.c_float * 3)(*target), up=(C.c_float * 3)(*up), fov_deg=fov, aspect=width / height,
                            near_=near, far_=far, width=width, height=height, light_dir=(C.c_float * 3)(*light_dir), ambient=ambient, diffuse=diffuse)
        ids = _i32(list(env_ids))
        rgba = np.zeros((len(ids), height, width, 4), dtype=np.uint8)
        depth = np.zeros((len(ids), height, width), dtype=np.float32)
        self._ck(self.lib.ag_render(self.h, C.byref(cam), len(ids), _p(ids), _p(rgba), _p(depth)))
        return rgba, depth

    # ---- fused dressing path
    def dressing_init(self, params, gender_is_male):
        self._dress_params = params
        self._ck(self.lib.ag_dressing_init(self.h, C.byref(params), _p(_i32(gender_is_male))))

    def dressing_set_tremor(self, on, rest, amplitude):
        self._ck(self.lib.ag_dressing_set_tremor(self.h, _p(_i32(on)), _p(_f32(rest, (self.n, 10))), _p(_f32(amplitude, (self.n, 10)))))

    def dressing_reset_episode(self, mask=None):
        self._ck(self.lib.ag_dressing_reset_episode(self.h, _p(_i32(mask))))

    def dressing_step_host(self, action):
        return self._step_host(self.lib.ag_dressing_step_host, 24, action)

    def dressing_step_dev(self, action_ptr, obs_ptr, reward_ptr, done_ptr, info_ptr):
        self._step_dev(self.lib.ag_dressing_step_dev, action_ptr, obs_ptr, reward_ptr, done_ptr, info_ptr)

    def feeding_reset_episode(self, mask=None):
        self._ck(self.lib.ag_feeding_reset_episode(self.h, _p(_i32(mask))))

    def feeding_step_host(self, action):
        return self._step_host(self.lib.ag_feeding_step_host, 25, action)

    def feeding_step_host_begin(self, action):
        self._ck(self.lib.ag_feeding_step_host_begin(self.h, _p(_f32(action, (self.n, 7)))))

    def feeding_step_host_end(self):
        return self._step_host(self.lib.ag_feeding_step_host_end, 25)

    def feeding_step_dev(self, action_ptr, obs_ptr, reward_ptr, done_ptr, info_ptr):
        self._step_dev(self.lib.ag_feeding_step_dev, action_ptr, obs_ptr, reward_ptr, done_ptr, info_ptr)


class BatchSimGroup:
    """One batch as G independent sub-batches, each a `BatchSim` on its own CUDA stream.

    Envs are independent (SURVEY.md 8(e)): nothing ties env A's sub-step to env B's except that a kernel launch covers
    the whole batch and ends with its slowest env -- in `k_pgs` the few envs that need all 50 sweeps keep a handful of
    warps busy for twice as long as the mean.  With the batch split into sub-batches that are enqueued back to back on
    separate streams, one sub-batch's tails are filled by the others' kernels.  The sub-batches are contiguous env
    ranges: entry points take whole-batch buffers and hand each sub-sim its slice."""

    def __init__(self, scene, cfg=None, n_envs=1, groups=1, device=0, _lib=None):
        if n_envs % groups:
            raise ValueError('n_envs must be a multiple of the number of sub-batches')
        self.n, self.groups, self.m = n_envs, groups, n_envs // groups
        self.sims = [BatchSim(scene, cfg, self.m, device=device, _lib=_lib) for _ in range(groups)]

    def slices(self):
        return [slice(g * self.m, (g + 1) * self.m) for g in range(self.groups)]

    def stream_ptrs(self):
        return [sim.stream_ptr() for sim in self.sims]

    def feeding_step_dev(self, action_ptr, obs_ptr, reward_ptr, done_ptr, info_ptr):
        """whole-batch device buffers ([n, 7], [n, 25], [n], [n], [n, 4] float32, contiguous); asynchronous"""
        for g, sim in enumerate(self.sims):
            o = 4 * g * self.m
            sim.feeding_step_dev(action_ptr + 7 * o, obs_ptr + 25 * o, reward_ptr + o, done_ptr + o, info_ptr + 4 * o)

    def feeding_step_host(self, action):
        a = _f32(action, (self.n, 7))
        for sl, sim in zip(self.slices(), self.sims):
            sim.feeding_step_host_begin(a[sl])
        parts = [sim.feeding_step_host_end() for sim in self.sims]
        return tuple(np.concatenate([p[k] for p in parts], axis=0) for k in range(4))

    def kernel_launches(self):
        return sum(sim.kernel_launches() for sim in self.sims)

    def overflow_count(self):
        return sum(sim.overflow_count() for sim in self.sims)

    def solver_stats(self):
        parts = [sim.solver_stats() for sim in self.sims]
        return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])

    def pgs_trips(self):
        parts = [sim.pgs_trips() for sim in self.sims]
        return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])

    def profile_enable(self, on=True):
        for sim in self.sims:
            sim.profile_enable(on)

    def profile_get(self):
        out = {}
        for sim in self.sims:
            for k, (ms, cnt) in sim.profile_get().items():
                a = out.get(k, (0.0, 0))
                out[k] = (a[0] + ms, a[1] + cnt)
        return out
