"""CPU tier of the headless renderer: the f110_view mirror against the C layout, argument validation of f110_render before any
CUDA call, the render kernels' resource usage, and hand-derived answers of the numpy restatement (oracle/render.py)."""
import ctypes
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from oracle import render as orender

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, 'include', 'f110_b200.h')


def test_f110_view_ctypes_layout_matches_c(tmp_path):
    from f1tenth_gym_b200 import _native as nat
    st = nat.F110View
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "%s"' % HEADER, 'int main(void){',
             'printf("size %zu\\n", sizeof(f110_view));']
    for f, _ in st._fields_:
        lines.append('printf("%s %%zu\\n", offsetof(f110_view, %s));' % (f, f))
    lines.append('return 0;}')
    src = tmp_path / 'view_layout.c'
    src.write_text('\n'.join(lines))
    exe = tmp_path / 'view_layout'
    subprocess.check_call(['gcc', '-o', str(exe), str(src)])
    out = dict(l.split() for l in subprocess.check_output([str(exe)]).decode().splitlines())
    assert int(out['size']) == ctypes.sizeof(st)
    for f, _ in st._fields_:
        assert int(out[f]) == getattr(st, f).offset, f


def _args():
    """A sim / view that pass validation without any device memory behind them (the pointers are never dereferenced on the
    host; validation returns before any CUDA call)."""
    from f1tenth_gym_b200 import _native as nat
    fake = 0x10000
    sim = nat.F110Sim()
    sim.num_envs, sim.num_agents, sim.integrator = 2, 2, 1
    sim.sim_length, sim.sim_width = 0.58, 0.31
    sim.state = fake
    view = nat.F110View()
    view.width, view.height, view.channels, view.camera, view.metres_per_pixel = 64, 48, 1, 1, 0.1
    return nat, sim, view, fake


def test_render_validates_before_any_cuda_call():
    nat, sim, view, fake = _args()
    L = nat.lib()
    assert 'f110_render' in nat.SIGNATURES and hasattr(L, 'f110_render')
    by = ctypes.byref
    empty_map = nat.F110Map()
    beams = nat.F110Beams()

    def call(s=sim, v=view, viewers=None, F=2, out=fake, m=empty_map):
        return L.f110_render(None if s is None else by(s), by(m), by(beams), None if v is None else by(v), viewers, F, out,
                             None, None)
    assert call() == -2                                  # no table bound: ValueError in Python, like the reference
    assert call(s=None) == -1 and call(v=None) == -1 and call(out=None) == -1
    assert call(out=fake + 1) == -1                      # output must allow 32-bit stores
    assert call(F=3) == -1                               # viewers NULL: one frame per env
    assert call(viewers=fake, F=0) == -1
    assert call(viewers=fake, F=5) == -2
    for field, bad in (('width', 62), ('width', 0), ('height', 0), ('channels', 2), ('camera', 2),
                       ('metres_per_pixel', 0.0), ('metres_per_pixel', float('nan')), ('draw_scan', 1),
                       ('num_waypoints', 3), ('num_waypoints', -1)):
        v = nat.F110View.from_buffer_copy(view)
        setattr(v, field, bad)
        assert call(v=v) == -1, (field, bad)
    v = nat.F110View.from_buffer_copy(view)
    v.table_start, v.num_tables = fake, 2            # planner layout without env_table
    assert call(v=v) == -1
    s = nat.F110Sim.from_buffer_copy(sim)
    s.sim_width = 0.0
    assert call(s=s) == -1
    with pytest.raises(ValueError):
        nat.check(-2)


def test_render_kernels_have_no_stack_beyond_the_trig_scratch():
    """No render kernel spills: their only stack is the 40-byte argument-reduction scratch of the fp64 sin / cos they share with
    f110_get_vertices (which the car test must match bit for bit), i.e. no more than k_vertices reserves."""
    from f1tenth_gym_b200 import _native as nat
    tool = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    if not os.path.exists(tool):
        pytest.skip('cuobjdump not available')
    nat.lib()
    out = subprocess.run([tool, '-res-usage', nat.LIB_PATH], capture_output=True, text=True).stdout
    usage = {fn: (int(reg), int(stack)) for fn, reg, stack in re.findall(r'Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+)', out)}
    vertices = [n for n in usage if '10k_vertices' in n]
    assert len(vertices) == 1, vertices
    trig = usage[vertices[0]][1]
    assert trig <= 40
    names = [n for n in usage if 'k_render_' in n]
    assert len(names) == 4, names        # k_render_frame<FAST = 0, 1>, k_render_scan, k_render_waypoints
    for n in names:
        assert usage[n][1] <= trig, (n, usage[n])


def _verts(x, y, hl, hw):
    """Axis-aligned car (yaw 0) in the rl, rr, fr, fl order of get_vertices."""
    return np.array([x - hl, y + hw, x - hl, y - hw, x + hl, y - hw, x + hl, y + hw])


def test_restatement_axis_aligned_cars():
    """mpp 0.125 puts pixel centres at odd multiples of 1/16 m: a 0.5 x 0.25 m car at the origin covers the centres
    x in {+-1/16, +-3/16}, y in {+-1/16}: 4 x 2 pixels.  A second car 0.25 m ahead covers x in {1/16, 3/16, 5/16, 7/16}; the
    viewer's car wins on the two shared columns, so the other car keeps 2 x 2 of its 4 x 2 pixels.  No map cell is a wall."""
    dt = np.ones((4, 4))
    W = H = 16
    lab = orender.base_labels((0.0, 0.0, 1.0, 0.0), W, H, 0.125, np.stack([_verts(0, 0, 0.25, 0.125), _verts(0.25, 0, 0.25, 0.125)]),
                              0, dt, 1.0, -100.0, -100.0, 1.0, 0.0)
    assert (lab == orender.VIEWER).sum() == 8
    assert (lab == orender.OTHER_CAR).sum() == 4
    rows, cols = np.nonzero(lab == orender.VIEWER)
    assert set(rows) == {7, 8} and set(cols) == {6, 7, 8, 9}
    assert set(np.nonzero(lab == orender.OTHER_CAR)[1]) == {10, 11}
    # the viewer's slot decides which car is label 2
    lab1 = orender.base_labels((0.0, 0.0, 1.0, 0.0), W, H, 0.125, np.stack([_verts(0, 0, 0.25, 0.125), _verts(0.25, 0, 0.25, 0.125)]),
                               1, dt, 1.0, -100.0, -100.0, 1.0, 0.0)
    assert (lab1 == orender.VIEWER).sum() == 8 and (lab1 == orender.OTHER_CAR).sum() == 4


def test_restatement_waypoint_pixel_heading_up():
    """Viewer at (2, 3) with yaw 0: camera 1 is (cx, cy, sin 0, -cos 0) = (2, 3, 0, -1).  A waypoint 1 m ahead and 0.5 m to the
    left, at 0.125 m per pixel in a 64 x 64 frame, is 8 rows above and 4 columns left of the centre: pixel (24, 28)."""
    cam = (2.0, 3.0, np.sin(0.0), -np.cos(0.0))
    lab = np.zeros((64, 64), dtype=np.uint8)
    orender.draw_points(lab, cam, 0.125, [3.0, 100.0], [3.5, 3.0], orender.WAYPOINT)
    assert list(zip(*np.nonzero(lab))) == [(24, 28)]          # the far point lands outside the frame and is dropped


def test_restatement_wall_cell_rotated_origin():
    """4 x 4 map, resolution 1, origin (10, 20, pi/2): x_rot = ty, y_rot = -tx, so cell (row 1, col 2) covers world
    x in (8, 9], y in [22, 23).  A 4 x 4 frame at 1 m per pixel centred on (8.25, 22.25) has pixel centres x in
    {6.75, 7.75, 8.75, 9.75}, y in {23.75, 22.75, 21.75, 20.75}: only pixel (row 1, col 2) is on the wall cell."""
    from f1tenth_gym_b200 import maps
    dt = np.ones((4, 4))
    dt[1, 2] = 0.0
    hm = maps.HostMap(dt, 1.0, (10.0, 20.0, np.pi / 2))
    lab = orender.base_labels((8.25, 22.25, 1.0, 0.0), 4, 4, 1.0, np.stack([_verts(50, 50, 0.25, 0.125)]), 0, hm.dt,
                              hm.resolution, hm.orig_x, hm.orig_y, hm.orig_c, hm.orig_s)
    expect = np.zeros((4, 4), dtype=np.uint8)
    expect[1, 2] = orender.WALL
    assert np.array_equal(lab, expect)
    # the same cell seen through walls() directly; points off the map are free, not dt[-1, -1]
    x = np.array([8.5, 9.5, 8.5, -50.0])
    y = np.array([22.5, 22.5, 21.5, -50.0])
    assert list(orender.walls(hm.dt, 1.0, hm.orig_x, hm.orig_y, hm.orig_c, hm.orig_s, x, y)) == [True, False, False, False]


def test_render_rejects_env_table_of_wrong_length():
    """The waypoint kernel reads env_table[env] for every env: a table per track instead of per env must be refused on the
    host, before anything reaches the device."""
    import torch
    import f1tenth_gym_b200 as f110
    cpu = torch.device('cpu')
    sim = f110.Simulator(f110.maps.DEFAULT_PARAMS, 1, 0, num_envs=6, device=cpu)
    tables = [np.stack([np.arange(4.0) + k, np.zeros(4), np.ones(4)], 1) for k in range(3)]
    pl = f110.PurePursuitPlanner(device=cpu, waypoints=tables, xind=0, yind=1, vind=2)
    view = f110.RenderView(64, 64, 0.1, channels=1).with_waypoints(pl, env_table=[0, 1, 2])
    with pytest.raises(ValueError, match='one table index per env'):
        sim.render(view)
    with pytest.raises(ValueError):
        f110.RenderView(64, 64, 0.1).with_waypoints(pl)             # a multi-table planner needs env_table
