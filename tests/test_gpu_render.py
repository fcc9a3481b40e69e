"""GPU tier of the headless renderer (C ABI f110_render, csrc/render.cuh): device frames against the numpy restatement
(oracle/render.py), fed the vertices of f110_get_vertices and the cameras the kernel reports in camera_out, so that labels must
match bit for bit; scan endpoints up to a 1e-9 px band at pixel edges (CUDA and numpy sin / cos may differ by an ulp)."""
import os

import numpy as np
import pytest
import torch

from oracle import render as orender

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, 'tests', 'golden')
MAPS = os.path.join(ROOT, 'f1tenth_gym_b200', 'maps')
EDGE = 1e-9


@pytest.fixture(scope='module')
def f110():
    import f1tenth_gym_b200 as f
    return f


@pytest.fixture(scope='module')
def dev():
    return torch.device('cuda:0')


def cpu(t):
    return t.detach().cpu().numpy()


def load_map(f110, dev, name):
    if name == 'rotated':
        k = np.load(os.path.join(G, 'scans_rotated_origin.npz'))
        hm0 = f110.maps.load_map(os.path.join(MAPS, 'example_map.yaml'), '.png')
        return f110.DeviceMap(f110.maps.HostMap(hm0.dt, float(k['resolution']), tuple(k['origin'])), dev)
    ext = '.pgm' if name == 'levine' else '.png'
    return f110.DeviceMap.from_yaml(os.path.join(MAPS, name + '.yaml'), ext, dev)


def near_wall_poses(dmap, N, A, rng, spacing=0.4):
    """Env e: agent 0 on a cell 0.1..0.35 m from a wall (its body overlaps the wall), agents 1.. `spacing` m behind it (the
    bodies overlap each other)."""
    h = dmap.host
    dt = cpu(dmap.dt) if dmap.dt.dim() == 2 else cpu(dmap.dt[0])
    r, c = np.nonzero((dt > 0.1) & (dt < 0.35))
    k = rng.integers(0, r.size, N)
    xr, yr = (c[k] + 0.5) * h.resolution, (r[k] + 0.5) * h.resolution
    x = h.orig_x + xr * h.orig_c - yr * h.orig_s
    y = h.orig_y + xr * h.orig_s + yr * h.orig_c
    yaw = rng.uniform(-np.pi, np.pi, N)
    poses = np.zeros((N, A, 3))
    for a in range(A):
        poses[:, a] = np.stack([x - a * spacing * np.cos(yaw), y - a * spacing * np.sin(yaw), yaw], 1)
    return poses


def all_vertices(f110, sim):
    st = sim.state
    poses = torch.stack([st[0], st[1], st[4]], 1).contiguous()
    v = f110.kernels.get_vertices(poses, sim.c.sim_length, sim.c.sim_width)
    return cpu(v).reshape(-1, 8)


def layer_dt(dmap, env, env_ids):
    if getattr(dmap, 'layers', None) is None:
        return dmap.host.dt if dmap.host.dt is not None else cpu(dmap.dt)
    return cpu(dmap.layers[int(env_ids[env])].dt)


def expected_base(f110, sim, view, viewers, cams, env_ids=None):
    """Labels 0-3 of every frame from the restatement."""
    N, A = sim.num_envs, sim.num_agents
    verts = all_vertices(f110, sim)
    h = sim.map.host
    out = np.zeros((len(viewers), view.height, view.width), dtype=np.uint8)
    for f, a in enumerate(viewers):
        if not 0 <= a < N * A:
            continue
        e = a // A
        out[f] = orender.base_labels(cams[f], view.width, view.height, view.metres_per_pixel, verts[e * A:(e + 1) * A], a % A,
                                     layer_dt(sim.map, e, env_ids), h.resolution, h.orig_x, h.orig_y, h.orig_c, h.orig_s)
    return out


def check_cameras(sim, view, viewers, cams):
    """camera_out, which the restatement is fed, against the definition: camera 0 = (center, 1, 0); camera 1 = (x, y, sin yaw,
    -cos yaw) of the viewer from `state` (CUDA and numpy sin / cos may differ by an ulp)."""
    if view.camera == 0:
        assert np.array_equal(cams, np.tile([view.center[0], view.center[1], 1.0, 0.0], (len(viewers), 1)))
        return
    st = cpu(sim.state)[:, viewers]
    assert np.array_equal(cams[:, :2], st[[0, 1]].T)
    ulp = np.spacing(1.0)
    assert np.all(np.abs(cams[:, 2] - np.sin(st[4])) <= ulp) and np.all(np.abs(cams[:, 3] + np.cos(st[4])) <= ulp)


def render_labels(sim, view, viewers):
    F = len(viewers)
    cams = torch.empty((F, 4), dtype=torch.float64, device=sim.device)
    out = sim.render(view, viewers=torch.as_tensor(viewers, dtype=torch.int32), camera_out=cams)
    return cpu(out)[..., 0], cpu(cams)


@pytest.mark.parametrize('name', ['example_map', 'berlin', 'levine', 'rotated'])
@pytest.mark.parametrize('A', [1, 2, 4])
def test_labels_match_restatement(f110, dev, name, A):
    """Both cameras; cars touching each other and walls after a few ticks; the ego, non-ego viewers and out-of-range ones."""
    dmap = load_map(f110, dev, name)
    N = 3
    rng = np.random.default_rng(A)
    sim = f110.Simulator(f110.maps.DEFAULT_PARAMS, A, 1, num_envs=N, device=dev)
    sim.set_device_map(dmap)
    sim.reset(near_wall_poses(dmap, N, A, rng))
    for _ in range(5):
        sim.step(np.stack([rng.uniform(-0.4, 0.4, (N, A)), rng.uniform(0, 3, (N, A))], 2))
    x0, y0 = float(sim.state[0, 0]), float(sim.state[1, 0])
    viewers = list(range(N * A)) + [-1, N * A, 2 ** 31 - 1]
    for view in (f110.RenderView(96, 80, 0.02, channels=1, camera=0, center=(x0, y0)),
                 f110.RenderView.follow(64, 0.025), f110.RenderView.follow(32, 0.1)):
        lab, cams = render_labels(sim, view, viewers)
        exp = expected_base(f110, sim, view, viewers, cams)
        assert np.array_equal(lab, exp), (name, A, view.camera, int((lab != exp).sum()))
        assert not lab[-3:].any() and not cams[-3:].any()            # out-of-range viewers: all-0 frame and camera
        check_cameras(sim, view, viewers[:N * A], cams[:N * A])
        if view.camera == 1:
            assert (lab[:N * A] == orender.VIEWER).any(axis=(1, 2)).all()      # the viewer's car is in view
    # the default viewers: one frame per env from its ego
    view = f110.RenderView.follow(64, 0.025)
    cams = torch.empty((N, 4), dtype=torch.float64, device=dev)
    lab = cpu(sim.render(view, camera_out=cams))[..., 0]
    assert np.array_equal(lab, expected_base(f110, sim, view, [e * A for e in range(N)], cpu(cams)))
    if A > 1:      # the touching cars and the walls both show up somewhere
        assert (lab == orender.OTHER_CAR).any() and (lab == orender.WALL).any()


def test_pure_pursuit_rollout_with_contacts(f110, dev):
    """example_map, 8 envs x 2 agents two waypoints apart, pure pursuit for 300 ticks (rear-end contacts and crashes), both
    cameras."""
    dmap = load_map(f110, dev, 'example_map')
    N, A = 8, 2
    sim = f110.Simulator(f110.maps.DEFAULT_PARAMS, A, 1, num_envs=N, device=dev)
    sim.set_device_map(dmap)
    wp = f110.maps.load_waypoints()
    ks = np.arange(N) * 90
    sim.reset(np.stack([np.stack([wp[k % len(wp)], wp[(k - 2) % len(wp)]]) for k in ks]))
    pl = f110.PurePursuitPlanner(device=dev)
    obs = sim.observations()
    contacts = 0.0
    for _ in range(300):
        obs = sim.step(pl.plan_actions(obs, 0.8, 1.3))
        contacts += float(sim.collisions.sum())
    assert contacts > 0
    viewers = list(range(N * A))
    for view in (f110.RenderView.follow(64, 0.02), f110.RenderView(128, 128, 0.2, channels=1, camera=0)):
        lab, cams = render_labels(sim, view, viewers)
        assert np.array_equal(lab, expected_base(f110, sim, view, viewers, cams))


def test_rgb_is_palette_of_labels(f110, dev):
    dmap = load_map(f110, dev, 'example_map')
    N, A = 2, 2
    sim = f110.Simulator(f110.maps.DEFAULT_PARAMS, A, 1, num_envs=N, device=dev, noise_std=0.0)
    sim.set_device_map(dmap)
    sim.reset(near_wall_poses(dmap, N, A, np.random.default_rng(0)))
    sim.step(np.zeros((N, A, 2)))
    pl = f110.PurePursuitPlanner(device=dev)
    pal = np.random.default_rng(1).integers(0, 256, (8, 3))
    for kw in (dict(), dict(palette=pal)):
        v1 = f110.RenderView.follow(64, 0.05, channels=1, draw_scan=True, **kw).with_waypoints(pl)
        v3 = f110.RenderView.follow(64, 0.05, channels=3, draw_scan=True, **kw).with_waypoints(pl)
        lab = cpu(sim.render(v1, viewers='all'))[..., 0]
        img = cpu(sim.render(v3, viewers='all'))
        assert img.shape == (N * A, 64, 64, 3) and img.dtype == np.uint8
        assert np.array_equal(img, v3.palette[lab])
        assert len(np.unique(lab)) >= 4
    ref = f110.render.REFERENCE_PALETTE
    assert ref[0] == (9, 32, 87) and ref[1] == (183, 193, 222) and ref[2] == (172, 97, 185) and ref[3] == (99, 52, 94)
    assert ref[5] == (183, 193, 222)


def test_stacked_maps_show_their_own_layer(f110, dev):
    from f1tenth_gym_b200 import trackgen as tg
    tracks = tg.random_tracks(1, 3)
    stacked, layers = tg.device_maps(tracks, dev)
    N, A = 6, 2
    ids = np.arange(N) % 3
    sim = f110.Simulator(f110.maps.DEFAULT_PARAMS, A, 1, num_envs=N, device=dev)
    sim.set_device_map(stacked, env_map_ids=ids)
    poses = np.zeros((N, A, 3))
    for e in range(N):
        t = tracks[ids[e]]
        for a in range(A):
            poses[e, a] = t.start_pose((20 * e - 5 * a) % t.waypoints.shape[0])
    sim.reset(poses)
    sim.step(np.zeros((N, A, 2)))
    view = f110.RenderView(128, 128, 0.5, channels=1, camera=0)
    viewers = [e * A for e in range(N)]
    lab, cams = render_labels(sim, view, viewers)
    assert np.array_equal(lab, expected_base(f110, sim, view, viewers, cams, env_ids=ids))
    walls = [lab[e] == orender.WALL for e in range(3)]
    assert not np.array_equal(walls[0], walls[1]) and not np.array_equal(walls[1], walls[2])
    assert np.array_equal(walls[0], lab[3] == orender.WALL)          # same layer, same walls


def test_waypoint_layer_single_and_per_env_tables(f110, dev):
    from f1tenth_gym_b200 import trackgen as tg
    # one table
    dmap = load_map(f110, dev, 'example_map')
    N, A = 3, 2
    sim = f110.Simulator(f110.maps.DEFAULT_PARAMS, A, 1, num_envs=N, device=dev)
    sim.set_device_map(dmap)
    wp = f110.maps.load_waypoints()
    sim.reset(np.stack([np.stack([wp[k], wp[k - 20]]) for k in (100, 300, 500)]))
    sim.step(np.zeros((N, A, 2)))
    pl = f110.PurePursuitPlanner(device=dev)
    wx, wy = cpu(pl.wx), cpu(pl.wy)
    viewers = list(range(N * A)) + [-1]
    for view in (f110.RenderView.follow(96, 0.1), f110.RenderView(200, 200, 0.5, channels=1, camera=0)):
        lab, cams = render_labels(sim, view.with_waypoints(pl), viewers)
        exp = expected_base(f110, sim, view, viewers, cams)
        for f in range(N * A):
            orender.draw_points(exp[f], cams[f], view.metres_per_pixel, wx, wy, orender.WAYPOINT)
        assert np.array_equal(lab, exp)
        assert (lab[:N * A] == orender.WAYPOINT).any(axis=(1, 2)).all() and not lab[-1].any()
    # per-env tables on stacked generated tracks
    tracks = tg.random_tracks(11, 3)
    stacked, _ = tg.device_maps(tracks, dev)
    N = 6
    ids = np.arange(N) % 3
    sim = f110.Simulator(f110.maps.DEFAULT_PARAMS, 1, 1, num_envs=N, device=dev)
    sim.set_device_map(stacked, env_map_ids=ids)
    sim.reset(np.stack([tracks[ids[e]].start_pose(30 * e)[None] for e in range(N)]))
    sim.step(np.zeros((N, 1, 2)))
    pl = f110.PurePursuitPlanner(device=dev, waypoints=[t.raceline() for t in tracks], xind=0, yind=1, vind=2)
    with pytest.raises(ValueError):
        f110.RenderView.follow(64, 0.1).with_waypoints(pl)
    short = f110.RenderView(160, 160, 0.5, channels=1, camera=0).with_waypoints(pl, env_table=[0, 1, 2])
    with pytest.raises(ValueError, match='one table index per env'):
        sim.render(short)
    view = f110.RenderView(160, 160, 0.5, channels=1, camera=0).with_waypoints(pl, env_table=ids)
    starts = cpu(pl.table_start)
    viewers = list(range(N))
    lab, cams = render_labels(sim, view, viewers)
    exp = expected_base(f110, sim, view, viewers, cams, env_ids=ids)
    for f in range(N):
        t = ids[f]
        rows = slice(starts[t], starts[t + 1])
        orender.draw_points(exp[f], cams[f], view.metres_per_pixel, cpu(pl.wx)[rows], cpu(pl.wy)[rows], orender.WAYPOINT)
    assert np.array_equal(lab, exp)


def test_scan_endpoints(f110, dev):
    dmap = load_map(f110, dev, 'example_map')
    N, A = 4, 2
    sim = f110.Simulator(f110.maps.DEFAULT_PARAMS, A, 1, num_envs=N, device=dev, noise_std=0.0, lidar_dist=0.1)
    sim.set_device_map(dmap)
    wp = f110.maps.load_waypoints()
    sim.reset(np.stack([np.stack([wp[k], wp[k - 30]]) for k in (50, 250, 450, 650)]))
    for _ in range(3):
        sim.step(np.tile([[0.1, 2.0]], (N, A, 1)))
    viewers = list(range(N * A))
    sp, ap = cpu(sim.scan_pose), cpu(sim.agent_poses)
    scans, angles = cpu(sim.scans), cpu(sim.beams.scan_angles)
    max_range = float(sim.map.c.max_range)
    for view in (f110.RenderView.follow(128, 0.05, draw_scan=True), f110.RenderView(256, 256, 0.1, channels=1, camera=0,
                                                                                       center=tuple(wp[50, :2]), draw_scan=True)):
        lab, cams = render_labels(sim, view, viewers)
        base = expected_base(f110, sim, view, viewers, cams)
        drawn_total = 0
        for f, a in enumerate(viewers):
            px, py = orender.scan_endpoints(sp[a, 0], sp[a, 1], ap[a, 2], angles, scans[a], max_range)
            r, c, inside, fr, fc = orender.point_pixels(cams[f], view.width, view.height, view.metres_per_pixel, px, py)
            drawn = lab[f] == orender.SCAN
            drawn_total += int(drawn.sum())
            # every drawn pixel is explained by an endpoint (within EDGE px of that pixel)
            for rr, cc in zip(*np.nonzero(drawn)):
                ok = (fr >= rr - EDGE) & (fr < rr + 1 + EDGE) & (fc >= cc - EDGE) & (fc < cc + 1 + EDGE)
                assert ok.any(), (f, rr, cc)
            # every endpoint farther than EDGE px from a pixel edge is drawn
            clear = inside & (np.abs(fr - np.rint(fr)) > EDGE) & (np.abs(fc - np.rint(fc)) > EDGE)
            assert drawn[r[clear], c[clear]].all(), f
            # and nothing else changed
            assert np.array_equal(lab[f][~drawn], base[f][~drawn])
        assert drawn_total > 100


def _rollout(f110, dev, render_every_tick):
    dmap = load_map(f110, dev, 'example_map')
    N, A = 16, 2
    sim = f110.Simulator(f110.maps.DEFAULT_PARAMS, A, 7, num_envs=N, device=dev, noise_std=0.01)
    sim.set_device_map(dmap)
    wp = f110.maps.load_waypoints()
    sim.env_reset(np.stack([np.stack([wp[k % 783], wp[(k - 3) % 783]]) for k in range(0, 16 * 45, 45)]))
    pl = f110.PurePursuitPlanner(device=dev)
    view = f110.RenderView.follow(64, 0.05, draw_scan=True).with_waypoints(pl)
    out = torch.empty(view.frame_shape(N * A), dtype=torch.uint8, device=dev)
    starts = torch.as_tensor(wp, device=dev).contiguous()
    obs = sim.observations()
    for _ in range(150):
        obs = sim.tick(pl.plan_actions(obs, 0.8, 1.4), autoreset_poses=starts)
        if render_every_tick:
            sim.render(view, viewers='all', out=out)
    return [cpu(t).copy() for t in (sim.state, sim.scans, sim.collisions, sim.lap_counts, sim.lap_times, sim.done)], sim, view


def test_no_side_effects_and_graph_capture(f110, dev):
    a, _, _ = _rollout(f110, dev, False)
    b, sim, view = _rollout(f110, dev, True)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    f1 = cpu(sim.render(view, viewers='all'))
    f2 = cpu(sim.render(view, viewers='all'))
    assert np.array_equal(f1, f2)
    # tick + render in one CUDA graph == the same calls made eagerly, on two identical simulators
    dmap = load_map(f110, dev, 'example_map')
    N, A = 8, 2
    wp = f110.maps.load_waypoints()
    poses = np.stack([np.stack([wp[k], wp[k - 3]]) for k in range(10, 8 * 90, 90)])
    sims, frames = [], []
    for _ in range(2):
        s = f110.Simulator(f110.maps.DEFAULT_PARAMS, A, 7, num_envs=N, device=dev, noise_std=0.01)
        s.set_device_map(dmap)
        s.env_reset(poses)
        sims.append(s)
        frames.append(torch.empty(view.frame_shape(N * A), dtype=torch.uint8, device=dev))
    actions = torch.tensor(np.tile([[0.05, 3.0]], (N * A, 1)), dtype=torch.float64, device=dev)
    viewers = torch.arange(N * A, dtype=torch.int32, device=dev)
    eager, graphed = sims
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):      # first-launch work outside the capture, on a throw-away simulator
        warm = f110.Simulator(f110.maps.DEFAULT_PARAMS, A, 7, num_envs=N, device=dev)
        warm.set_device_map(dmap)
        warm.env_reset(poses)
        warm.tick(actions)
        warm.render(view, viewers=viewers, out=torch.empty_like(frames[1]))
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize(dev)
    with torch.cuda.graph(g):
        graphed.tick(actions)
        graphed.render(view, viewers=viewers, out=frames[1])
    for _ in range(20):
        eager.tick(actions)
        eager.render(view, viewers=viewers, out=frames[0])
        g.replay()
        torch.cuda.synchronize(dev)
        assert torch.equal(frames[0], frames[1])
        assert torch.equal(eager.state, graphed.state)


def test_env_render(f110, dev):
    wp = f110.maps.load_waypoints()
    env = f110.F110Env(map='example_map', num_agents=2, scan_noise_std=0.0)
    env.reset(np.stack([wp[0], wp[-15]]))
    img = env.render('rgb_array')
    assert isinstance(img, np.ndarray) and img.shape == (800, 1000, 3) and img.dtype == np.uint8
    assert np.array_equal(img, cpu(env.sim.render(f110.RenderView.reference()))[0])
    assert 'rgb_array' in f110.F110Env.metadata['render.modes']
    with pytest.raises(NotImplementedError):
        env.render('human')
    with pytest.raises(NotImplementedError):
        env.render()
    benv = f110.F110Env(map='example_map', num_agents=2, num_envs=4, scan_noise_std=0.0)
    benv.reset(np.stack([np.stack([wp[k], wp[k - 15]]) for k in (0, 200, 400, 600)]))
    one = benv.render('rgb_array')
    assert one.is_cuda and tuple(one.shape) == (1, 800, 1000, 3)
    two = benv.render('rgb_array', env_ids=[1, 3])
    assert torch.equal(two, benv.sim.render(f110.RenderView.reference(), viewers=[2, 6]))
    assert torch.equal(one[0], benv.sim.render(f110.RenderView.reference())[0])
    small = benv.render('rgb_array', view=f110.RenderView.follow(64, 0.05, channels=3), env_ids=[2])
    assert tuple(small.shape) == (1, 64, 64, 3)


def test_per_agent_frames_cfg3_size(f110, dev):
    """16384 envs x 2 agents: one 64 x 64 heading-up label frame per agent (32768 frames); 64 random frames against the
    restatement."""
    dmap = load_map(f110, dev, 'example_map')
    N, A = 16384, 2
    sim = f110.Simulator(f110.maps.DEFAULT_PARAMS, A, 1, num_envs=N, device=dev)
    sim.set_device_map(dmap)
    wp = f110.maps.load_waypoints()
    k = np.arange(N) % len(wp)
    sim.reset(np.stack([wp[k], wp[(k - 3) % len(wp)]], 1))
    sim.step(np.tile([[0.05, 2.0]], (N, A, 1)))
    view = f110.RenderView.follow(64, 0.05)
    cams = torch.empty((N * A, 4), dtype=torch.float64, device=dev)
    out = sim.render(view, viewers='all', camera_out=cams)
    assert tuple(out.shape) == (N * A, 64, 64, 1)
    pick = np.random.default_rng(0).choice(N * A, 64, replace=False)
    lab = cpu(out[torch.as_tensor(pick, device=dev)])[..., 0]
    exp = expected_base(f110, sim, view, list(pick), cpu(cams)[pick])
    assert np.array_equal(lab, exp)
