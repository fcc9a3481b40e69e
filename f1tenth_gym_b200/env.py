"""F110Env façade — the gym.Env-shaped surface of reference f110_env.py:53-418, batched.

    env = F110Env(map=..., map_ext='.png', num_agents=2, timestep=0.01, integrator=Integrator.RK4,
                  num_envs=4096)                       # num_envs is the batch extension
    obs, reward, done, info = env.reset(poses)         # poses (A,3) or (N,A,3); runs ONE zero-action tick
    obs, reward, done, info = env.step(action)         # action (N,A,2) = (steer, speed)

kwargs and defaults are the reference's (f110_env.py:104-159): seed=12345, map='vegas', map_ext='.png',
params=<18-key dict>, num_agents=2, timestep=0.01, ego_idx=0, integrator=RK4, lidar_dist=0.0.
Extensions: num_envs (None = single env, reference-shaped numpy/list outputs; int = batched torch
tensors (N,A,...) that are views of device buffers valid until the next step), num_beams, fov, device,
scan_noise_std (reference default 0.01; 0 disables the noise for bit-reproducible parity runs).
The gym 0.19 API with the non-standard reset(poses) is kept on purpose (SURVEY.md 8b).
render(mode='rgb_array') draws top-down frames on the device (render.py); there is no 'human' window.
"""
import numpy as np
import torch

from . import maps as hostmaps
from .simulator import Integrator, Simulator


class F110Env(object):
    metadata = {'render.modes': ['human', 'human_fast', 'rgb_array']}
    render_callbacks = []

    def __init__(self, **kwargs):
        self.seed = kwargs.get('seed', 12345)
        if 'map' in kwargs:
            self.map_name = kwargs['map']
            self.map_path = hostmaps.resolve_map_path(self.map_name)
        else:
            self.map_name = 'vegas'
            self.map_path = hostmaps.resolve_map_path('vegas')
        self.map_ext = kwargs.get('map_ext', '.png')
        self.params = kwargs.get('params', dict(hostmaps.DEFAULT_PARAMS))
        self.num_agents = kwargs.get('num_agents', 2)
        self.timestep = kwargs.get('timestep', 0.01)
        self.ego_idx = kwargs.get('ego_idx', 0)
        self.integrator = kwargs.get('integrator', Integrator.RK4)
        self.lidar_dist = kwargs.get('lidar_dist', 0.0)
        num_envs = kwargs.get('num_envs', None)
        self.batched = num_envs is not None
        self.num_envs = int(num_envs) if self.batched else 1
        self.start_thresh = 0.5
        self.sim = Simulator(self.params, self.num_agents, self.seed, time_step=self.timestep,
                             ego_idx=self.ego_idx, integrator=self.integrator, lidar_dist=self.lidar_dist,
                             num_envs=self.num_envs, num_beams=kwargs.get('num_beams', 1080),
                             fov=kwargs.get('fov', 4.7), device=kwargs.get('device', None),
                             noise_std=kwargs.get('scan_noise_std', 0.01))
        self.sim.set_map(self.map_path, self.map_ext)
        self.render_obs = None
        # single-env mode: the whole observation comes back in ONE batch of async copies + one stream sync
        # (C ABI f110_step_host) instead of a blocking .cpu() per field
        self._io = None if self.batched else self.sim.make_host_io()

    # env-level state lives on the device (f110_env.py:165-189); expose the reference's attribute names
    @property
    def lap_times(self):
        return self._out(self.sim.lap_times)

    @property
    def lap_counts(self):
        return self._out(self.sim.lap_counts)

    @property
    def toggle_list(self):
        return self._out(self.sim.toggle_list)

    @property
    def current_time(self):
        return self.sim.current_time if self.batched else float(self.sim.current_time[0].item())

    @property
    def collisions(self):
        return self._out(self.sim.collisions)

    def _out(self, t):
        t = t.view(self.num_envs, self.num_agents)
        return t if self.batched else t[0].cpu().numpy()

    def _finish(self, obs):
        sim = self.sim
        sim.env_post_step()
        N, A = self.num_envs, self.num_agents
        if self.batched:
            obs['lap_times'] = sim.lap_times.view(N, A)
            obs['lap_counts'] = sim.lap_counts.view(N, A)
            done = sim.done.bool()
            info = {'checkpoint_done': sim.checkpoint_done.view(N, A).bool()}
            return obs, self.timestep, done, info
        # single-env, reference-shaped (base_classes.py:594-612): lists of per-agent values
        o = {'ego_idx': obs['ego_idx'],
             'scans': [s for s in obs['scans'][0].double().cpu().numpy()],
             'collisions': obs['collisions'][0].cpu().numpy(),
             'lap_times': sim.lap_times.cpu().numpy(), 'lap_counts': sim.lap_counts.cpu().numpy()}
        for k in ('poses_x', 'poses_y', 'poses_theta', 'linear_vels_x', 'linear_vels_y', 'ang_vels_z'):
            o[k] = [float(v) for v in obs[k][0].cpu().numpy()]
        done = bool(sim.done[0].item())
        info = {'checkpoint_done': sim.checkpoint_done.bool().cpu().numpy()}
        return o, self.timestep, done, info

    def _step_single(self, action):
        """Reference-shaped step of ONE env (base_classes.py:594-612 obs dict of per-agent lists): actions go through a
        pinned buffer, f110_step_host runs step + lap logic and copies scans / state / collisions / done / laps back."""
        sim, io, A = self.sim, self._io, self.num_agents
        a = np.asarray(action.cpu() if torch.is_tensor(action) else action, dtype=np.float64).reshape(A, 2)
        io['actions'].numpy()[:] = a
        sim.step_host(io)
        st = io['state'].numpy()                      # [7][A]
        lap_counts = io['lap_counts'].numpy().copy()
        o = {'ego_idx': self.ego_idx,
             'scans': [s for s in io['scans'].numpy().astype(np.float64)],
             'poses_x': [float(v) for v in st[0]], 'poses_y': [float(v) for v in st[1]],
             'poses_theta': [float(v) for v in st[4]], 'linear_vels_x': [float(v) for v in st[3]],
             'linear_vels_y': [0.0] * A, 'ang_vels_z': [float(v) for v in st[5]],
             'collisions': io['collisions'].numpy().copy(),
             'lap_times': io['lap_times'].numpy().copy(), 'lap_counts': lap_counts}
        # toggle_list >= 4 (f110_env.py:243) <=> lap_counts = floor(toggle / 2) >= 2
        return o, self.timestep, bool(io['done'].numpy()[0]), {'checkpoint_done': lap_counts >= 2}

    def step(self, action):
        """f110_env.py:263-304."""
        if not self.batched:
            return self._step_single(action)
        obs = self.sim.step(action)
        return self._finish(obs)

    def reset(self, poses):
        """f110_env.py:306-349: zero counters, start frame, Simulator.reset, then ONE zero-action tick
        whose (obs, reward, done, info) is returned."""
        self.sim.env_reset(poses)
        action = torch.zeros((self.num_envs, self.num_agents, 2), dtype=torch.float64, device=self.sim.device)
        return self.step(action)

    def reset_envs(self, env_mask, poses):
        """Batch extension: re-initialise only the masked envs (counters + Simulator.reset); no tick is run."""
        self.sim.env_reset(poses, env_mask)

    def update_map(self, map_path, map_ext):
        """f110_env.py:351-362"""
        self.sim.set_map(map_path, map_ext)

    def update_params(self, params, index=-1):
        """f110_env.py:364-375"""
        self.sim.update_params(params, agent_idx=index)

    def add_render_callback(self, callback_func):
        """f110_env.py:377-385 (kept for API compatibility; the callbacks expect a pyglet EnvRenderer and are not called by
        render('rgb_array'))."""
        F110Env.render_callbacks.append(callback_func)

    def render(self, mode='human', view=None, env_ids=None):
        """f110_env.py:387-418.  mode='rgb_array' draws top-down frames on the device (render.RenderView, default the
        reference window: 1000x800, fixed camera at the origin), each env seen from its ego: single-env mode returns an
        (H, W, 3) uint8 numpy array, batched mode a (len(env_ids), H, W, 3) uint8 CUDA tensor of the envs env_ids (default
        (0,): a reference-size frame is 2.4 MB).  'human' / 'human_fast' windows are not available."""
        assert mode in F110Env.metadata['render.modes']
        if mode != 'rgb_array':
            raise NotImplementedError('f1tenth_gym_b200 has no renderer (pyglet/OpenGL GUI is out of scope).')
        from .render import RenderView
        view = RenderView.reference() if view is None else view
        if not self.batched:
            return self.sim.render(view)[0].cpu().numpy()
        ids = torch.as_tensor((0,) if env_ids is None else env_ids, dtype=torch.int64).reshape(-1)
        if ids.numel() == 0 or int(ids.min()) < 0 or int(ids.max()) >= self.num_envs:
            raise ValueError('env_ids must be env indices in [0, %d)' % self.num_envs)
        return self.sim.render(view, viewers=ids * self.num_agents + self.ego_idx)
