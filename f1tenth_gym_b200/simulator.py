"""Batched Simulator: the host-side mirror of reference base_classes.py (Simulator / RaceCar) for
N independent environments x A agents stepped in lockstep by the CUDA path.

Mirrors the reference interface for this path — same constructor arguments, method names, argument
meaning and error behaviour:
    Simulator(params, num_agents, seed, time_step=0.01, ego_idx=0, integrator=Integrator.RK4,
              lidar_dist=0.0)                                   base_classes.py:465-497
    .set_map(map_path, map_ext)                                 :499-511
    .update_params(params, agent_idx=-1)   IndexError           :514-534
    .reset(poses)                           ValueError           :614-630
    .step(control_inputs) -> observations dict                  :553-612
plus the batch extensions `num_envs`, `num_beams`, `fov`, `device`, `noise_std`.

PyTorch is used only as the device-memory allocator and stream provider; all compute goes through
the C ABI in libf110_b200.so (include/f110_b200.h).  There is no CPU fallback.
"""
import ctypes as C
from enum import Enum

import numpy as np
import torch

from . import _native as nat
from . import maps as hostmaps


class Integrator(Enum):     # base_classes.py:40-42
    RK4 = 1
    Euler = 2


def _stream_ptr(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class DeviceMap(object):
    """ScanSimulator2D state (laser_models.py:348-427) resident in HBM: fp64 DT grid + angle LUTs."""

    def __init__(self, host_map, device, theta_dis=2000, eps=0.0001, max_range=30.0, _device_dt=None):
        self.host = host_map
        self.device = device
        self.theta_dis = theta_dis
        sines, cosines = hostmaps.angle_lut(theta_dis)
        # cell-unit copy for the fast path (res = 2^-k: the division is an exact exponent shift)
        self.dt_cells = self.dt_codes = self.dt_lut = self.dt_cells_pad = self.dt_codes_pad = None
        if _device_dt is not None:
            self.dt = _device_dt
            if host_map.fast_path:
                self.dt_cells = self.dt / host_map.resolution     # IEEE fp64 division on the device, exact here
        else:
            self.dt = torch.from_numpy(host_map.dt).to(device)
            if host_map.fast_path:
                cells = host_map.dt / host_map.resolution
                codes, lut = hostmaps.code_table(cells)
                self.dt_cells = torch.from_numpy(cells).to(device)
                self.dt_codes = torch.from_numpy(codes).to(device)
                self.dt_lut = torch.from_numpy(lut).to(device)
                self.dt_codes_pad = self._pad(self.dt_codes, pitch_multiple=16)
        if self.dt_cells is not None:
            self.dt_cells_pad = self._pad(self.dt_cells)
        self.sines = torch.from_numpy(sines).to(device)
        self.cosines = torch.from_numpy(cosines).to(device)
        sc = np.ascontiguousarray(np.stack([sines, cosines], axis=1))
        self.sincos = torch.from_numpy(sc).to(device)
        self.sincos2 = torch.from_numpy(np.ascontiguousarray(np.concatenate([sc, sc], axis=0))).to(device)
        # smallest positive DT value (= resolution for an exact EDT): the lean march kernel tests `d != 0` for `d > eps`
        pos = self.dt[self.dt > 0]
        dt_min_positive = float(pos.min().item()) if pos.numel() else float('inf')
        self.c = nat.F110Map(host_map.height, host_map.width, host_map.resolution, host_map.orig_x,
                             host_map.orig_y, host_map.orig_c, host_map.orig_s, eps, max_range, theta_dis,
                             host_map.fast_path, host_map.dt_oob, nat.ptr(self.dt), nat.ptr(self.dt_cells),
                             nat.ptr(self.dt_codes), nat.ptr(self.dt_lut), nat.ptr(self.sines), nat.ptr(self.cosines),
                             nat.ptr(self.sincos), nat.ptr(self.dt_cells_pad), nat.ptr(self.dt_codes_pad),
                             0 if self.dt_codes_pad is None else self.dt_codes_pad.shape[1],
                             nat.ptr(self.sincos2), dt_min_positive, 1)

    @staticmethod
    def _pad(t, pitch_multiple=1):
        """[H][W] -> [H+1][W+1 rounded up to pitch_multiple] with the extra row / columns holding t[-1,-1] (what an
        off-map lookup reads)."""
        H, W = t.shape
        Wp = -(-(W + 1) // pitch_multiple) * pitch_multiple
        out = torch.empty((H + 1, Wp), dtype=t.dtype, device=t.device)
        out[:] = t[-1, -1]
        out[:H, :W] = t
        return out.contiguous()

    @classmethod
    def stack(cls, maps):
        """Multi-map batch (SURVEY 8f row 3): several DeviceMaps that share size, resolution and origin are
        stacked into one [L][H][W] table; Simulator.set_device_map(stacked, env_map_ids) picks one per env."""
        m0 = maps[0]
        for m in maps[1:]:
            h, h0 = m.host, m0.host
            if (h.height, h.width, h.resolution, h.orig_x, h.orig_y, h.orig_c, h.orig_s) != \
               (h0.height, h0.width, h0.resolution, h0.orig_x, h0.orig_y, h0.orig_c, h0.orig_s):
                raise ValueError('stacked maps must share size, resolution and origin')
        out = cls.__new__(cls)
        out.__dict__.update(m0.__dict__)
        out.layers = list(maps)
        out.dt = torch.stack([m.dt for m in maps]).contiguous()
        out.dt_cells = torch.stack([m.dt_cells for m in maps]).contiguous() if m0.dt_cells is not None else None
        out.dt_cells_pad = torch.stack([m.dt_cells_pad for m in maps]).contiguous() if m0.dt_cells_pad is not None else None
        out.dt_codes = out.dt_lut = out.dt_codes_pad = None
        c = nat.F110Map.from_buffer_copy(m0.c)
        c.dt = nat.ptr(out.dt)
        c.dt_cells = nat.ptr(out.dt_cells)
        c.dt_cells_pad = nat.ptr(out.dt_cells_pad)
        c.dt_codes = None
        c.dt_lut = None
        c.dt_codes_pad = None
        c.num_layers = len(maps)
        c.dt_min_positive = min(m.c.dt_min_positive for m in maps)
        out.c = c
        return out

    @classmethod
    def from_device_dt(cls, dt, resolution, origin, **kw):
        """A map whose fp64 distance table [H][W] (metres) already lives on the device (e.g. rasterised track +
        f110_edt): nothing but the out-of-bounds scalar dt[-1,-1] crosses PCIe."""
        dt = dt.contiguous()
        meta = hostmaps.HostMap.meta(dt.shape[0], dt.shape[1], resolution, origin, float(dt[-1, -1].item()))
        return cls(meta, dt.device, _device_dt=dt, **kw)

    @classmethod
    def from_yaml(cls, map_path, map_ext, device, edt='scipy', **kw):
        """edt='scipy': the reference's host pipeline; edt='device': C ABI f110_edt (bit-identical table)."""
        if edt == 'device':
            return cls(hostmaps.load_map_device_edt(map_path, map_ext, device), device, **kw)
        return cls(hostmaps.load_map(map_path, map_ext), device, **kw)


class DeviceBeams(object):
    """Per-beam tables of RaceCar.__init__ (base_classes.py:122-158) in HBM."""

    def __init__(self, num_beams, fov, params, device, theta_dis=2000):
        self.num_beams, self.fov = num_beams, fov
        sa, co, sd = hostmaps.beam_tables(num_beams, fov, params)
        self.scan_angles = torch.from_numpy(sa).to(device)
        self.cosines = torch.from_numpy(co).to(device)
        self.side_distances = torch.from_numpy(sd).to(device)
        self.cos_side = torch.from_numpy(np.ascontiguousarray(np.stack([co, sd], axis=1))).to(device)
        self.angle_increment = fov / (num_beams - 1)
        self.c = nat.F110Beams(num_beams, fov, self.angle_increment,
                               hostmaps.theta_index_increment(num_beams, fov, theta_dis),
                               nat.ptr(self.scan_angles), nat.ptr(self.cosines), nat.ptr(self.side_distances),
                               nat.ptr(self.cos_side), float(sd.max()))


def empty_map_struct():
    """A map struct with no DT bound: stepping with it raises ValueError like the reference
    (laser_models.py:445-446 'Map is not set for scan simulator.')."""
    return nat.F110Map()


class Simulator(object):
    """N x A batched simulator.  All state lives in persistent device buffers (SoA over the flat agent
    index a = env*A + agent); the observation tensors returned by step() are VIEWS of those buffers
    and are overwritten by the next step (the reference likewise returns aliases of internal arrays,
    base_classes.py:594-602)."""

    def __init__(self, params, num_agents, seed, time_step=0.01, ego_idx=0, integrator=Integrator.RK4,
                 lidar_dist=0.0, num_envs=1, num_beams=1080, fov=4.7, device=None, noise_std=0.0,
                 count_lookups=False, march_queue=True, march_item_beams=32):
        nat.lib()   # fail loudly right away if the CUDA library is missing
        if device is None:
            device = torch.device('cuda', torch.cuda.current_device())
        self.device = torch.device(device)
        self.num_agents = int(num_agents)
        self.num_envs = int(num_envs)
        self.seed = seed
        self.time_step = time_step
        self.ego_idx = ego_idx
        self.params = params
        self.integrator = integrator
        self.lidar_dist = lidar_dist
        self.num_beams, self.fov = num_beams, fov
        if isinstance(integrator, Integrator):
            integ = integrator.value
        elif integrator in (1, 2):
            integ = int(integrator)
        else:
            name = getattr(integrator, 'name', integrator)
            raise SyntaxError("Invalid Integrator Specified. Provided %s. Please choose RK4 or Euler" % name)
        N, A, B = self.num_envs, self.num_agents, num_beams
        NA = N * A
        dev = self.device
        f64 = dict(dtype=torch.float64, device=dev)
        i32 = dict(dtype=torch.int32, device=dev)
        self.params_dev = torch.from_numpy(np.tile(hostmaps.params_vector(params), (A, 1))).to(dev)
        self.state = torch.zeros((7, NA), **f64)
        self.steer_buf = torch.zeros((2, NA), **f64)
        self.steer_cnt = torch.zeros((NA,), **i32)
        self.scan_pose = torch.zeros((NA, 4), **f64)
        self.agent_poses = torch.zeros((NA, 5), **f64)
        self.scans = torch.zeros((NA, B), dtype=torch.float32, device=dev)
        self.wall_flag = torch.zeros((NA,), **i32)
        self.collisions = torch.zeros((NA,), **f64)
        self.collision_idx = torch.full((NA,), -1, **i32)
        # F110Env-level arrays (f110_env.py:165-189), batched
        self.current_time = torch.zeros((N,), **f64)
        self.lap_times = torch.zeros((NA,), **f64)
        self.lap_counts = torch.zeros((NA,), **f64)
        self.toggle_list = torch.zeros((NA,), **f64)
        self.near_starts = torch.ones((NA,), **i32)
        self.start_xs = torch.zeros((NA,), **f64)
        self.start_ys = torch.zeros((NA,), **f64)
        self.start_thetas = torch.zeros((NA,), **f64)
        self.start_rot = torch.eye(2, **f64).reshape(1, 4).repeat(N, 1).contiguous()
        self.done = torch.zeros((N,), dtype=torch.uint8, device=dev)
        self.checkpoint_done = torch.zeros((NA,), dtype=torch.uint8, device=dev)
        self.env_arrivals = torch.zeros((N,), **i32)
        self.lookup_counter = torch.zeros((1,), dtype=torch.int64, device=dev) if count_lookups else None
        self.tick_counter = torch.zeros((1,), dtype=torch.int64, device=dev)
        # work queue of the persistent ray-march kernel (csrc/march.cuh): last tick's heavy items go first
        ib = int(march_item_beams)
        assert ib in (32, 64)
        self.march_ipa = (B + ib - 1) // ib if (march_queue and (B + ib - 1) // ib <= 256) else 0
        items = NA * self.march_ipa
        self.march_cost = torch.full((NA * 256,), -1, **i32) if self.march_ipa else None
        self.march_order = torch.zeros((3, items), **i32) if self.march_ipa else None
        self.march_count = torch.zeros((4,), **i32) if self.march_ipa else None
        self.march_rec = torch.zeros((NA, 8), **f64) if self.march_ipa else None
        self.beams = DeviceBeams(num_beams, fov, params, dev)
        self.map = None
        self._map_struct = empty_map_struct()
        self._actions_dev = torch.zeros((NA, 2), **f64)
        self.c = nat.F110Sim(
            N, A, integ, ego_idx, 0, time_step, lidar_dist, 0.005, float(params['length']), float(params['width']),
            nat.ptr(self.params_dev), nat.ptr(self.state), nat.ptr(self.steer_buf), nat.ptr(self.steer_cnt),
            nat.ptr(self.scan_pose), nat.ptr(self.agent_poses), nat.ptr(self.scans), nat.ptr(self.wall_flag),
            nat.ptr(self.collisions), nat.ptr(self.collision_idx), nat.ptr(self.current_time),
            nat.ptr(self.lap_times), nat.ptr(self.lap_counts), nat.ptr(self.toggle_list),
            nat.ptr(self.near_starts), nat.ptr(self.start_xs), nat.ptr(self.start_ys),
            nat.ptr(self.start_thetas), nat.ptr(self.start_rot), nat.ptr(self.done),
            nat.ptr(self.checkpoint_done), nat.ptr(self.env_arrivals), None, nat.ptr(self.lookup_counter), nat.ptr(self.tick_counter),
            nat.ptr(self.march_cost), nat.ptr(self.march_order), nat.ptr(self.march_count), self.march_ipa,
            nat.ptr(self.march_rec), float(noise_std), int(seed) & 0xFFFFFFFFFFFFFFFF)
        self._graph = None
        self._render_all = None      # viewers='all' of render(): every flat agent index, made on first use
        self._zeros_NA = torch.zeros((N, A), dtype=torch.float64, device=dev)     # obs['linear_vels_y'] (always 0, :606)

    # ------------------------------------------------------------------ configuration
    def set_map(self, map_path, map_ext, edt='scipy'):
        """base_classes.py:499-511 / laser_models.py:383-427 (load-time: PIL + yaml + EDT; edt='device' runs the
        exact distance transform on the GPU instead of scipy on the host)."""
        self.set_device_map(DeviceMap.from_yaml(map_path, map_ext, self.device, edt=edt))

    def set_device_map(self, device_map, env_map_ids=None):
        """env_map_ids (N,) ints: which layer of a DeviceMap.stack() each env uses (multi-map batches)."""
        self.map = device_map
        self._map_struct = device_map.c
        self._graph = None
        layers = getattr(device_map.c, 'num_layers', 1)
        if layers > 1:
            ids = torch.zeros((self.num_envs,), dtype=torch.int32) if env_map_ids is None else \
                torch.as_tensor(env_map_ids, dtype=torch.int32)
            if ids.numel() != self.num_envs or int(ids.min()) < 0 or int(ids.max()) >= layers:
                raise ValueError('env_map_ids must hold num_envs layer indices in [0, %d)' % layers)
            self.env_layer = ids.to(self.device).contiguous()
            self.c.env_layer = nat.ptr(self.env_layer)
        else:
            self.env_layer = None
            self.c.env_layer = None

    def update_params(self, params, agent_idx=-1, env_mask=None):
        """base_classes.py:514-534.  agent_idx < 0: every agent slot; else that slot (in every env).
        Batch extension: env_mask (N,) bool restricts the update to those envs — the parameter table then
        becomes per env ([N*A][18], dynamics randomisation); `params` may also be a (N, 18) / (N, A, 18) tensor
        of per-env parameter vectors (key order maps.PARAM_KEYS)."""
        if not (agent_idx < 0 or 0 <= agent_idx < self.num_agents):
            raise IndexError('Index given is out of bounds for list of agents.')
        N, A = self.num_envs, self.num_agents
        per_env_values = not isinstance(params, dict)
        if env_mask is None and not per_env_values and not self.c.params_per_env:
            pv = torch.from_numpy(hostmaps.params_vector(params)).to(self.device)
            if agent_idx < 0:
                self.params_dev[:] = pv
            else:
                self.params_dev[agent_idx] = pv
            return
        if not self.c.params_per_env:        # expand the shared table once
            self.params_dev = self.params_dev.unsqueeze(0).repeat(N, 1, 1).contiguous()
            self.c.params = nat.ptr(self.params_dev)
            self.c.params_per_env = 1
            self._graph = None
        if per_env_values:
            pv = torch.as_tensor(params, dtype=torch.float64).to(self.device)
            pv = pv.reshape(N, -1, 18)                        # (N,1,18) broadcasts over agents, or (N,A,18)
        else:
            pv = torch.from_numpy(hostmaps.params_vector(params)).to(self.device).reshape(1, 1, 18)
        m = torch.ones((N,), dtype=torch.bool, device=self.device) if env_mask is None else \
            torch.as_tensor(env_mask).to(device=self.device, dtype=torch.bool)
        tgt = self.params_dev if agent_idx < 0 else self.params_dev[:, agent_idx:agent_idx + 1]
        src = pv if (agent_idx < 0 or pv.shape[1] == 1) else pv[:, agent_idx:agent_idx + 1]
        tgt[m] = src.expand(N, tgt.shape[1], 18)[m]

    def set_noise(self, std_dev, seed=None):
        """Scan noise N(0, std_dev^2) (laser_models.py:429,450-452); 0 disables (parity runs)."""
        self.c.noise_std = float(std_dev)
        if seed is not None:
            self.c.noise_seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        self._graph = None

    # ------------------------------------------------------------------ helpers
    def _poses_tensor(self, poses):
        N, A = self.num_envs, self.num_agents
        p = torch.as_tensor(poses, dtype=torch.float64)
        if p.dim() == 2:
            if p.shape[0] != A:
                raise ValueError('Number of poses for reset does not match number of agents.')
            p = p.unsqueeze(0).expand(N, A, 3)
        elif p.dim() != 3 or p.shape[0] != N or p.shape[1] != A:
            raise ValueError('Number of poses for reset does not match number of agents.')
        return p.to(self.device).contiguous()

    def _actions_tensor(self, control_inputs):
        N, A = self.num_envs, self.num_agents
        a = control_inputs
        if not (torch.is_tensor(a) and a.is_cuda and a.dtype == torch.float64 and a.is_contiguous()
                and a.numel() == N * A * 2):
            a = torch.as_tensor(np.asarray(a) if not torch.is_tensor(a) else a, dtype=torch.float64)
            if a.dim() == 2 and N > 1:
                a = a.unsqueeze(0).expand(N, A, 2)
            if a.numel() != N * A * 2:
                raise ValueError('control_inputs must have shape (num_envs, num_agents, 2)')
            self._actions_dev.copy_(a.reshape(N * A, 2), non_blocking=True)
            a = self._actions_dev
        return a

    def _mask_ptr(self, env_mask):
        if env_mask is None:
            return None, None
        m = torch.as_tensor(env_mask).to(device=self.device, dtype=torch.uint8).contiguous()
        if m.numel() != self.num_envs:
            raise ValueError('env_mask must have num_envs entries')
        return m, nat.ptr(m)

    # ------------------------------------------------------------------ reference-surface methods
    def reset(self, poses, env_mask=None):
        """Simulator.reset (base_classes.py:614-630): zero state, place agents, empty steer FIFO.
        poses: (A,3) broadcast to every env, or (N,A,3).  env_mask (N,) bool: partial reset."""
        p = self._poses_tensor(poses)
        m, mp = self._mask_ptr(env_mask)
        nat.check(nat.lib().f110_reset(C.byref(self.c), nat.ptr(p), mp, _stream_ptr(self.device)))

    def env_reset(self, poses, env_mask=None):
        """Counters and start frame of F110Env.reset (f110_env.py:319-331) + Simulator.reset."""
        p = self._poses_tensor(poses)
        m, mp = self._mask_ptr(env_mask)
        L = nat.lib()
        nat.check(L.f110_env_reset(C.byref(self.c), nat.ptr(p), mp, _stream_ptr(self.device)))
        nat.check(L.f110_reset(C.byref(self.c), nat.ptr(p), mp, _stream_ptr(self.device)))

    def step(self, control_inputs):
        """Simulator.step (base_classes.py:553-612). control_inputs (N,A,2) = (steer, speed)."""
        a = self._actions_tensor(control_inputs)
        nat.check(nat.lib().f110_step(C.byref(self.c), C.byref(self._map_struct), C.byref(self.beams.c),
                                      nat.ptr(a), _stream_ptr(self.device)))
        return self.observations()

    def env_post_step(self):
        """Tail of F110Env.step: time + lap logic + done (f110_env.py:294-302, 204-246)."""
        nat.check(nat.lib().f110_env_post_step(C.byref(self.c), _stream_ptr(self.device)))

    def autoreset(self, start_poses, pose_gap=23, seed=12345):
        """Reset every env whose ego collided to a hashed draw from start_poses (device (K,3) fp64)."""
        nat.check(nat.lib().f110_autoreset(C.byref(self.c), nat.ptr(start_poses), start_poses.shape[0],
                                           pose_gap, int(seed), 0, _stream_ptr(self.device)))

    def tick(self, control_inputs, env_level=True, autoreset_poses=None, pose_gap=23, seed=12345):
        """One whole tick in three launches (C ABI f110_tick): step + lap logic + optional auto-reset, same
        results as step(); env_post_step(); autoreset()."""
        a = self._actions_tensor(control_inputs)
        n = 0 if autoreset_poses is None else autoreset_poses.shape[0]
        nat.check(nat.lib().f110_tick(C.byref(self.c), C.byref(self._map_struct), C.byref(self.beams.c), nat.ptr(a),
                                      1 if env_level else 0, nat.ptr(autoreset_poses), n, pose_gap, int(seed),
                                      _stream_ptr(self.device)))
        return self.observations()

    def observations(self):
        N, A, B = self.num_envs, self.num_agents, self.num_beams
        st = self.state
        return {'ego_idx': self.ego_idx,
                'scans': self.scans.view(N, A, B),
                'poses_x': st[0].view(N, A), 'poses_y': st[1].view(N, A), 'poses_theta': st[4].view(N, A),
                'linear_vels_x': st[3].view(N, A),
                'linear_vels_y': self._zeros_NA,
                'ang_vels_z': st[5].view(N, A),
                'collisions': self.collisions.view(N, A)}

    # ------------------------------------------------------------------ throughput paths
    def capture_graph(self, actions, autoreset_poses=None, pose_gap=23, autoreset_seed=12345, env_level=False):
        """Capture one tick (f110_step [+ env_post_step] [+ autoreset]) reading `actions` (a persistent
        device tensor the caller overwrites between replays) into a CUDA graph.  The warm-up tick that precedes the
        capture runs on a snapshot: every simulation buffer (state, FIFO, scans, lap counters, tick counter / noise
        stream, march queue history) is restored afterwards, so capturing has no side effect on the simulation."""
        assert actions.is_cuda and actions.dtype == torch.float64 and actions.is_contiguous()
        L = nat.lib()
        names = ('state', 'steer_buf', 'steer_cnt', 'scan_pose', 'agent_poses', 'scans', 'wall_flag', 'collisions',
                 'collision_idx', 'current_time', 'lap_times', 'lap_counts', 'toggle_list', 'near_starts', 'start_xs',
                 'start_ys', 'start_thetas', 'start_rot', 'done', 'checkpoint_done', 'tick_counter', 'march_cost',
                 'march_order', 'march_count', 'march_rec')
        snapshot = {n: getattr(self, n).clone() for n in names if getattr(self, n, None) is not None}

        def tick():
            n = 0 if autoreset_poses is None else autoreset_poses.shape[0]
            nat.check(L.f110_tick(C.byref(self.c), C.byref(self._map_struct), C.byref(self.beams.c), nat.ptr(actions),
                                  1 if env_level else 0, nat.ptr(autoreset_poses), n, pose_gap, int(autoreset_seed),
                                  _stream_ptr(self.device)))
        side = torch.cuda.Stream(self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            tick()      # warm-up outside capture (module load, first-launch work)
        torch.cuda.current_stream(self.device).wait_stream(side)
        torch.cuda.synchronize(self.device)
        for n, t in snapshot.items():
            getattr(self, n).copy_(t)
        torch.cuda.synchronize(self.device)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            tick()
        self._graph = g
        self._graph_keep = (actions, autoreset_poses)
        return g

    def replay(self):
        self._graph.replay()

    def make_host_io(self, with_scans=True, packed_scans=False):
        """Pinned host buffers for step_host() / step_host_async().  packed_scans=True (async path only): the scan block
        crosses PCIe as 24-bit fixed point (io['scans_u24'] uint8 [NA, B, 3]; decode with unpack_scans_u24) instead of fp32."""
        N, A, B = self.num_envs, self.num_agents, self.num_beams
        NA = N * A
        if packed_scans:
            with_scans = False
        io = {'actions': torch.zeros((NA, 2), dtype=torch.float64).pin_memory(),
              'scans': torch.zeros((NA, B), dtype=torch.float32).pin_memory() if with_scans else None,
              'scans_u24': torch.zeros((NA, B, 3), dtype=torch.uint8).pin_memory() if packed_scans else None,
              'state': torch.zeros((7, NA), dtype=torch.float64).pin_memory(),
              'collisions': torch.zeros((NA,), dtype=torch.float64).pin_memory(),
              'done': torch.zeros((N,), dtype=torch.uint8).pin_memory(),
              'lap_times': torch.zeros((NA,), dtype=torch.float64).pin_memory(),
              'lap_counts': torch.zeros((NA,), dtype=torch.float64).pin_memory()}
        io['_struct'] = nat.F110HostObs(nat.ptr(io['scans']), nat.ptr(io['state']), nat.ptr(io['collisions']),
                                        nat.ptr(io['done']), nat.ptr(io['lap_times']), nat.ptr(io['lap_counts']),
                                        nat.ptr(io['scans_u24']))
        return io

    @staticmethod
    def unpack_scans_u24(buf):
        """uint8 [..., 3] (io['scans_u24']) -> float32 ranges: (b0 | b1 << 8 | b2 << 16) * 2^-19 m."""
        b = (buf.numpy() if torch.is_tensor(buf) else np.asarray(buf)).astype(np.uint32)
        return ((b[..., 0] | (b[..., 1] << 8) | (b[..., 2] << 16)).astype(np.float32) * np.float32(2.0 ** -19))

    def step_host(self, io):
        """One tick through HOST buffers (C ABI f110_step_host): H2D actions, step, env_post_step,
        D2H observation, stream sync.  io from make_host_io(); fill io['actions'] first."""
        nat.check(nat.lib().f110_step_host(C.byref(self.c), C.byref(self._map_struct), C.byref(self.beams.c),
                                           nat.ptr(io['actions']), nat.ptr(self._actions_dev),
                                           C.byref(io['_struct']), _stream_ptr(self.device)))
        return io

    def make_host_pipeline(self, depth=2, with_scans=True, packed_scans=False):
        """`depth` independent sets of (pinned host obs, device staging, events, actions scratch) for
        step_host_async(); one shared copy stream."""
        N, A, B = self.num_envs, self.num_agents, self.num_beams
        NA = N * A
        dev = self.device
        copy_stream = torch.cuda.Stream(dev)
        sets = []
        if packed_scans:
            with_scans = False
        for _ in range(depth):
            io = self.make_host_io(with_scans, packed_scans)
            st = {'scans': torch.zeros((NA, B), dtype=torch.float32, device=dev) if with_scans else None,
                  'scans_u24': torch.zeros((NA, B, 3), dtype=torch.uint8, device=dev) if packed_scans else None,
                  'state': torch.zeros((7, NA), dtype=torch.float64, device=dev),
                  'collisions': torch.zeros((NA,), dtype=torch.float64, device=dev),
                  'done': torch.zeros((N,), dtype=torch.uint8, device=dev),
                  'lap_times': torch.zeros((NA,), dtype=torch.float64, device=dev),
                  'lap_counts': torch.zeros((NA,), dtype=torch.float64, device=dev)}
            io['_stage'] = st
            io['_stage_struct'] = nat.F110HostObs(nat.ptr(st['scans']), nat.ptr(st['state']), nat.ptr(st['collisions']),
                                                  nat.ptr(st['done']), nat.ptr(st['lap_times']), nat.ptr(st['lap_counts']),
                                                  nat.ptr(st['scans_u24']))
            io['_actions_dev'] = torch.zeros((NA, 2), dtype=torch.float64, device=dev)
            io['_ev_tick'] = torch.cuda.Event()
            io['_ev_copy'] = torch.cuda.Event()
            io['_ev_tick'].record()
            io['_ev_copy'].record()
            io['_copy_stream'] = copy_stream
            sets.append(io)
        torch.cuda.synchronize(dev)
        return sets

    def step_host_async(self, io):
        """Enqueue one tick whose observation lands in io's pinned host buffers (C ABI f110_step_host_async);
        returns immediately.  Call wait_host(io) before reading them or before reusing io."""
        nat.check(nat.lib().f110_step_host_async(
            C.byref(self.c), C.byref(self._map_struct), C.byref(self.beams.c), nat.ptr(io['actions']),
            nat.ptr(io['_actions_dev']), C.byref(io['_stage_struct']), C.byref(io['_struct']),
            _stream_ptr(self.device), C.c_void_p(io['_copy_stream'].cuda_stream),
            C.c_void_p(io['_ev_tick'].cuda_event), C.c_void_p(io['_ev_copy'].cuda_event)))
        return io

    @staticmethod
    def wait_host(io):
        io['_ev_copy'].synchronize()

    def step_profile(self, control_inputs):
        """One tick with CUDA events around each kernel -> (dynamics_ms, raymarch_ms, finalize_ms)."""
        a = self._actions_tensor(control_inputs)
        ms = (C.c_float * 3)()
        nat.check(nat.lib().f110_step_profile(C.byref(self.c), C.byref(self._map_struct), C.byref(self.beams.c),
                                              nat.ptr(a), ms, _stream_ptr(self.device)))
        return float(ms[0]), float(ms[1]), float(ms[2])

    def render(self, view, viewers=None, out=None, camera_out=None):
        """Top-down frames of the current state on the device (render.py, C ABI f110_render): returns `out`, a uint8 CUDA tensor
        (F, H, W, channels), allocated only when out is None.  viewers: None = one frame per env from its ego_idx, 'all' = one
        per flat agent index env*A + agent, or F flat agent indices (an out-of-range index gives an all-0 frame).
        camera_out (F, 4) fp64, optional, receives each frame's (cx, cy, cr, sr).  No host synchronisation."""
        from . import render
        if isinstance(viewers, str) and viewers == 'all':
            if self._render_all is None:
                self._render_all = torch.arange(self.num_envs * self.num_agents, dtype=torch.int32, device=self.device)
            viewers = self._render_all
        return render.render(self, view, viewers, out, camera_out)

    def lookups(self):
        return int(self.lookup_counter.item()) if self.lookup_counter is not None else None
