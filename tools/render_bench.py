"""Timing of the headless renderer (f110_render) on one GPU; writes one JSON file.

    python tools/render_bench.py [--out profiles/render/render_bench.json] [--iters 300]

Workloads
  (a) cfg3 state (16384 envs x 2 agents, example_map): one 64 x 64 heading-up label frame per agent = 32768 frames per call;
  (b) 16 reference-size RGB frames (1000 x 800, fixed camera, 0.024 m per pixel);
  (c) one CUDA graph holding f110_tick + (a), against a graph holding the tick alone: what (a) adds per tick.
Each time is CUDA events around `iters` warmed back-to-back launches (the frames, 134 MB for (a), 38 MB for (b), are written
once per call; the inputs are the state and the 20 MB distance table, so the map stays L2-resident, as in a training loop).
Bytes are what the frames hold; the share of bandwidth is against 7.7 TB/s (data-sheet HBM3e bandwidth of one B200).  A sample
of each workload's frames is checked against the numpy restatement (oracle/render.py) at that size.  GPU name and power limit
are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import f1tenth_gym_b200 as f110             # noqa: E402
from oracle import render as orender        # noqa: E402

PEAK_BW = 7.7e12


def gpu_info():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in q.split(',')]
        return {'gpu': name, 'power_limit': power, 'max_sm_clock': clock}
    except Exception as e:      # the measurement itself still stands; say what is missing
        return {'gpu': torch.cuda.get_device_name(0), 'power_limit': 'unknown (%s)' % e}


def time_us(fn, iters, warmup=20):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / iters


def check_sample(sim, view, viewers, frames, cams, k, seed):
    """k random frames of a label render against the restatement (labels 0-3)."""
    N, A = sim.num_envs, sim.num_agents
    st = sim.state
    verts = f110.kernels.get_vertices(torch.stack([st[0], st[1], st[4]], 1).contiguous(), sim.c.sim_length, sim.c.sim_width)
    verts = verts.cpu().numpy().reshape(-1, 8)
    h = sim.map.host
    pick = np.random.default_rng(seed).choice(len(viewers), k, replace=False)
    bad = 0
    for f in pick:
        a = int(viewers[f])
        e = a // A
        exp = orender.base_labels(cams[f], view.width, view.height, view.metres_per_pixel, verts[e * A:(e + 1) * A], a % A,
                                  h.dt, h.resolution, h.orig_x, h.orig_y, h.orig_c, h.orig_s)
        bad += int(not np.array_equal(frames[f], exp))
    return {'frames_checked': int(k), 'frames_mismatched': bad}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'render', 'render_bench.json'))
    ap.add_argument('--iters', type=int, default=300)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('render_bench: no CUDA device')
    dev = torch.device('cuda:0')
    res = {'info': gpu_info(), 'iters': args.iters}
    dmap = f110.DeviceMap.from_yaml(f110.maps.resolve_map_path('example_map'), '.png', dev)
    wp = f110.maps.load_waypoints()
    N, A = 16384, 2
    sim = f110.Simulator(f110.maps.DEFAULT_PARAMS, A, 12345, num_envs=N, device=dev, noise_std=0.0)
    sim.set_device_map(dmap)
    k = np.arange(N) % len(wp)
    sim.env_reset(np.stack([wp[k], wp[(k - 23) % len(wp)]], 1))
    actions = torch.tensor(np.tile([[0.05, 3.0]], (N * A, 1)), dtype=torch.float64, device=dev)
    for _ in range(5):
        sim.tick(actions)
    torch.cuda.synchronize()

    # (a) one 64 x 64 label frame per agent
    va = f110.RenderView.follow(64, 0.05)
    viewers = torch.arange(N * A, dtype=torch.int32, device=dev)
    out_a = torch.empty(va.frame_shape(N * A), dtype=torch.uint8, device=dev)
    cams_a = torch.empty((N * A, 4), dtype=torch.float64, device=dev)
    us = time_us(lambda: sim.render(va, viewers=viewers, out=out_a), args.iters)
    nbytes = out_a.numel()
    res['a_per_agent_64x64_labels'] = {
        'frames': N * A, 'us_per_call': us, 'bytes_written': nbytes, 'GB_per_s': nbytes / us * 1e-3,
        'share_of_7.7TB_per_s': nbytes / (us * 1e-6) / PEAK_BW}
    sim.render(va, viewers=viewers, out=out_a, camera_out=cams_a)
    res['a_per_agent_64x64_labels']['check'] = check_sample(sim, va, viewers.cpu().numpy(), out_a.cpu().numpy()[..., 0],
                                                            cams_a.cpu().numpy(), 64, 0)

    # (b) 16 reference-size RGB frames
    vb = f110.RenderView.reference()
    vb_lab = f110.RenderView(1000, 800, 1.2 / 50, channels=1, camera=0)
    vw = torch.arange(0, 16 * A, A, dtype=torch.int32, device=dev)
    out_b = torch.empty(vb.frame_shape(16), dtype=torch.uint8, device=dev)
    us = time_us(lambda: sim.render(vb, viewers=vw, out=out_b), args.iters)
    nbytes = out_b.numel()
    res['b_reference_rgb_1000x800'] = {
        'frames': 16, 'us_per_call': us, 'bytes_written': nbytes, 'GB_per_s': nbytes / us * 1e-3,
        'share_of_7.7TB_per_s': nbytes / (us * 1e-6) / PEAK_BW}
    cams_b = torch.empty((16, 4), dtype=torch.float64, device=dev)
    lab_b = sim.render(vb_lab, viewers=vw, camera_out=cams_b).cpu().numpy()[..., 0]
    chk = check_sample(sim, vb_lab, vw.cpu().numpy(), lab_b, cams_b.cpu().numpy(), 4, 1)
    chk['rgb_equals_palette_of_labels'] = bool(np.array_equal(out_b.cpu().numpy(), vb.palette[lab_b]))
    res['b_reference_rgb_1000x800']['check'] = chk

    # (c) tick + (a) in one graph against the tick alone
    def capture(with_render):
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            sim.tick(actions)
            if with_render:
                sim.render(va, viewers=viewers, out=out_a)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize()
        with torch.cuda.graph(g):
            sim.tick(actions)
            if with_render:
                sim.render(va, viewers=viewers, out=out_a)
        return g
    g_tick, g_both = capture(False), capture(True)
    rounds = []
    for _ in range(3):          # alternate the two graphs; the host is shared with other work
        t0 = time_us(g_tick.replay, args.iters)
        t1 = time_us(g_both.replay, args.iters)
        rounds.append((t0, t1))
    t_tick = float(np.median([r[0] for r in rounds]))
    t_both = float(np.median([r[1] for r in rounds]))
    res['c_graph_tick_plus_a'] = {'tick_us': t_tick, 'tick_plus_render_us': t_both, 'render_adds_us': t_both - t_tick,
                                  'rounds_us': rounds}
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == '__main__':
    main()
