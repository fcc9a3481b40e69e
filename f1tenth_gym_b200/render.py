"""Headless renderer: top-down frames drawn on the device (C ABI f110_render, csrc/render.cuh), no window and no GL.

    view = RenderView.reference()                     # the reference window: 1000x800 RGB, fixed camera at the origin
    frames = sim.render(view, viewers=[0, 5])         # (2, 800, 1000, 3) uint8 CUDA tensor
    obs = sim.render(RenderView.follow(64, 0.1), viewers='all')   # (N*A, 64, 64, 1) labels, heading up, one per agent

Labels (channels=1) and their default colours (channels=3, the reference's rendering.py / waypoint_follow.py colours):
    0 free or off the map  (9, 32, 87)        1 wall              (183, 193, 222)
    2 the viewer's car      (172, 97, 185)     3 other cars        (99, 52, 94)
    4 scan endpoints        (255, 255, 255)    5 waypoints         (183, 193, 222)
Walls fill the map cells the simulator collides with (dt == 0, image pixels <= 128); the reference draws 1-pixel points at
the corners of the 0-valued image pixels instead.  Text labels, 'human' windows and pyglet render callbacks are not drawn.
"""
import ctypes as C

import numpy as np

from . import _native as nat

# reference colours: glClearColor and the map points / ego car / other cars of rendering.py, waypoints of waypoint_follow.py;
# scan endpoints have no reference counterpart (white)
REFERENCE_PALETTE = ((9, 32, 87), (183, 193, 222), (172, 97, 185), (99, 52, 94), (255, 255, 255), (183, 193, 222),
                     (0, 0, 0), (0, 0, 0))
FREE, WALL, VIEWER, OTHER_CAR, SCAN, WAYPOINT = range(6)


class RenderView(object):
    """What a frame shows: size, channels (1 = label, 3 = RGB), camera (0 = fixed window centred on `center`, 1 = centred on
    the viewer with its heading up), metres per pixel, the scan-endpoint layer and an optional waypoint layer."""

    def __init__(self, width, height, metres_per_pixel, channels=3, camera=0, center=(0.0, 0.0), draw_scan=False,
                 palette=REFERENCE_PALETTE):
        if width <= 0 or height <= 0 or width % 4 != 0:
            raise ValueError('width must be a positive multiple of 4 and height positive')
        if channels not in (1, 3) or camera not in (0, 1) or not metres_per_pixel > 0:
            raise ValueError('channels must be 1 or 3, camera 0 or 1, metres_per_pixel > 0')
        pal = np.asarray(palette, dtype=np.uint8)
        if pal.shape != (8, 3):
            raise ValueError('palette must hold 8 RGB triples')
        self.width, self.height, self.channels, self.camera = int(width), int(height), int(channels), int(camera)
        self.metres_per_pixel = float(metres_per_pixel)
        self.center = (float(center[0]), float(center[1]))
        self.draw_scan = bool(draw_scan)
        self.palette = pal
        self.planner = self.env_table = None      # keep the device tables the struct points into alive
        self.c = nat.F110View(self.width, self.height, self.channels, self.camera, self.center[0], self.center[1],
                              self.metres_per_pixel, int(self.draw_scan))
        for i in range(8):
            for k in range(3):
                self.c.palette[i][k] = int(pal[i, k])

    @classmethod
    def reference(cls, **kw):
        """The reference window (f110_env.py:50-51 WINDOW_W/H, rendering.py zoom 1.2 at 50 px/m): 1000x800 RGB, camera 0 at
        (0, 0), 0.024 m per pixel, reference colours."""
        return cls(1000, 800, 1.2 / 50, channels=3, camera=0, center=(0.0, 0.0), **kw)

    @classmethod
    def follow(cls, size, metres_per_pixel, channels=1, **kw):
        """size x size frame centred on the viewer, heading up (camera 1): the bird's-eye policy input."""
        return cls(size, size, metres_per_pixel, channels=channels, camera=1, **kw)

    def with_waypoints(self, planner, env_table=None):
        """Draw a PurePursuitPlanner's waypoints (its device tables are reused).  A multi-table planner needs env_table, the
        (num_envs,) table index of each env, as for plan_actions(table_ids=...)."""
        import torch
        self.c.wx, self.c.wy, self.c.num_waypoints = nat.ptr(planner.wx), nat.ptr(planner.wy), planner.wx.shape[0]
        self.c.table_start, self.c.num_tables, self.c.env_table = None, 0, None
        if planner.table_start is not None:
            if env_table is None:
                raise ValueError('this planner holds %d waypoint tables: pass env_table' % planner.num_tables)
            et = torch.as_tensor(env_table).to(device=planner.device, dtype=torch.int32).reshape(-1).contiguous()
            self.c.table_start, self.c.num_tables, self.c.env_table = nat.ptr(planner.table_start), planner.num_tables, nat.ptr(et)
            self.env_table = et
        else:
            if env_table is not None:
                raise ValueError('env_table given with a single-table planner')
            self.env_table = None
        self.planner = planner
        return self

    def frame_shape(self, num_frames):
        return (num_frames, self.height, self.width, self.channels)


def _on(t, dev):
    """t lives on the simulator's device (a device given as plain 'cuda' means the one current when it was built)."""
    return t.is_cuda and (dev.index is None or t.device.index == dev.index)


def render(sim, view, viewers=None, out=None, camera_out=None):
    """Simulator.render: see there (viewers: None or flat agent indices)."""
    import torch
    dev = sim.device
    N, A = sim.num_envs, sim.num_agents
    if viewers is None:
        vt, F = None, N
    else:
        if isinstance(viewers, str):
            raise ValueError("viewers must be None, 'all' or flat agent indices")
        vt = torch.as_tensor(viewers)
        if vt.dtype != torch.int32:      # wider indices saturate, so that an out-of-range one stays out of range
            vt = vt.to(torch.int64).clamp(-1, 2 ** 31 - 1)
        vt = vt.to(device=dev, dtype=torch.int32).reshape(-1).contiguous()
        F = vt.numel()
        if F == 0:
            raise ValueError('no viewers given')
    if view.env_table is not None and view.env_table.numel() != N:
        # the kernel reads env_table[env] for every env of the batch
        raise ValueError('env_table must hold one table index per env (%d), not %d' % (N, view.env_table.numel()))
    if view.planner is not None and not _on(view.planner.wx, dev):
        raise ValueError('the waypoint tables must live on the simulator\'s device %s' % dev)
    shape = view.frame_shape(F)
    if out is None:
        out = torch.empty(shape, dtype=torch.uint8, device=dev)
    elif not (_on(out, dev) and out.dtype == torch.uint8 and out.is_contiguous() and tuple(out.shape) == shape):
        raise ValueError('out must be a contiguous uint8 tensor on %s of shape %s' % (dev, shape))
    if camera_out is not None and not (_on(camera_out, dev) and camera_out.dtype == torch.float64 and
                                       camera_out.is_contiguous() and tuple(camera_out.shape) == (F, 4)):
        raise ValueError('camera_out must be a contiguous float64 tensor on %s of shape (%d, 4)' % (dev, F))
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    nat.check(nat.lib().f110_render(C.byref(sim.c), C.byref(sim._map_struct), C.byref(sim.beams.c), C.byref(view.c),
                                    nat.ptr(vt), F, nat.ptr(out), nat.ptr(camera_out), stream))
    return out
