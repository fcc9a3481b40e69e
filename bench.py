#!/usr/bin/env python
"""bench.py — agent-steps/sec of the batched F1TENTH hot path on N B200s (weak scaling), with the
roofline of the ray-march kernel and the CPU baseline beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg3|cfg2|cfg2x2|cfg5_B] [--no-extras]
    python bench.py ... --dump-outputs DIR    # also write the last timed tick's observation as DIR/<name>.npy
    python bench.py --impl reference ...      # the reference's own numba path (oracle/_ref), one process per host core
    torchrun ... bench.py --gpus N ...        # one rank per GPU; envs shard, no data-path collective

A "step" is one tick (Simulator.step + F110Env lap logic + auto-reset) over the workload's whole env
batch on each GPU.  `value` = agent-steps/s over all GPUs with inputs resident in HBM, timed with CUDA
events per step (L2 flushed between steps, outside the event pairs), max over ranks.  `e2e` = the same
metric through the host-buffer API (f110_step_host_async): pinned H2D of the actions and D2H of the full
observation (scans, state, collisions, done, laps) inside the timed region, every step.

The default workload is BASELINE.json configs[2] (16384 envs x 2 agents, GJK + opponent ray-cast live), which is
also the per-GPU share of configs[3] (131072 x 2 over 8 GPUs), so `--gpus 8` IS configs[3].  On one GPU the same
run also measures configs[1] (4096 x 1), the north_star's 4096 x 2 and the configs[4] beam sweep with fewer steps and
reports them under `workloads` (value, ms_per_step, e2e, roofline each).  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the tree may be read-only: the benchmark writes nothing into it

import numpy as np  # noqa: E402


def _baseline_metric():
    """The metric string is BASELINE.json's, verbatim."""
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'BASELINE.json')) as f:
            return json.load(f)['metric']
    except Exception:
        return 'agent-steps/sec (1080-beam scan) at 1/2/4/8 B200 vs reference numba CPU'


METRIC = _baseline_metric()
UNIT = 'agent-steps/s'
WORKLOADS = {
    # BASELINE.json configs[1]
    'cfg2': dict(num_envs=4096, num_agents=1, num_beams=1080,
                 desc='4096 single-agent envs, example_map, 1080 beams, random actions (BASELINE configs[1])'),
    # the north_star target sentence: 4096 envs x 2 agents
    'cfg2x2': dict(num_envs=4096, num_agents=2, num_beams=1080,
                   desc='4096 envs x 2 agents, example_map, 1080 beams, random actions (north_star target)'),
    # BASELINE.json configs[2]; 8 ranks of it are configs[3]
    'cfg3': dict(num_envs=16384, num_agents=2, num_beams=1080,
                 desc='16384 envs x 2 agents with GJK, example_map, 1080 beams (BASELINE configs[2]; per-GPU share of configs[3])'),
}
for _b in (270, 540, 1080, 2160):
    WORKLOADS['cfg5_%d' % _b] = dict(num_envs=32768, num_agents=1, num_beams=_b,
                                     desc='beam sweep: 32768 single-agent envs, %d beams (BASELINE configs[4])' % _b)
DEFAULT_WORKLOAD = 'cfg3'
EXTRA_WORKLOADS = ['cfg2', 'cfg2x2', 'cfg5_270', 'cfg5_540', 'cfg5_1080', 'cfg5_2160']
POSE_GAP = 23          # second agent 23 waypoints (~4.6 m) behind (SURVEY 8d)
SEED = 12345
FLUSH_BYTES = 256 << 20
DUMP_SCAN_BYTES = 48 << 20      # --dump-outputs: scan rows beyond this are sampled (the whole dump stays under 64 MB)
DUMP_SEED = 2024


def config_dict(workload, world, sample=None):
    """The `config` object: the same keys and values for the CUDA arm and the reference arm."""
    w = WORKLOADS[workload]
    return {'workload': workload, 'description': w['desc'], 'map': 'example_map (1600x1600, 0.0625 m)',
            'num_envs_per_gpu': w['num_envs'], 'num_agents': w['num_agents'], 'num_beams': w['num_beams'],
            'integrator': 'RK4', 'timestep': 0.01, 'scan_noise': 'off',
            'actions': 'steer~U[-0.4189,0.4189], speed~U[0,8] i.i.d. per tick',
            'auto_reset': 'ego collision -> fresh start pose on the raceline',
            'parallelism': 'env-sharded x%d, no collective' % world}


def measured_peak():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    try:
        with open(p) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


def ncu_traffic(workload):
    """dram bytes per march-kernel launch from the committed ncu capture summary, if one exists for this workload."""
    p = os.path.join(ROOT, 'profiles', 'raymarch_ncu_summary.json')
    try:
        with open(p) as f:
            d = json.load(f)
        return d.get(workload, {}).get('dram_bytes_per_launch')
    except Exception:
        return None


def pci_bus_id(gpu_index):
    """PCI bus id ('0000:1b:00.0') of CUDA device `gpu_index` (honours CUDA_VISIBLE_DEVICES, unlike an NVML index)."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(gpu_index)
        return '%04x:%02x:%02x.0' % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
    except Exception:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(gpu_index)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        return bus[4:] if len(bus.split(':')[0]) == 8 else bus      # NVML prints an 8-digit domain, sysfs a 4-digit one


def numa_bind(gpu_index):
    """Pin this rank to the CPUs of its GPU's NUMA node BEFORE any pinned allocation: cudaHostAlloc places the pages
    where the calling thread runs, and a D2H into the far socket's memory costs a third of the PCIe rate (round 1,
    8 GPUs: 52 -> 38 GB/s per GPU)."""
    info = {'bound': False}
    try:
        bus = pci_bus_id(gpu_index)
        info['pci'] = bus
        with open('/sys/bus/pci/devices/%s/numa_node' % bus) as f:
            node = int(f.read().strip())
        info['gpu_numa_node'] = node
        if node < 0:
            return info
        with open('/sys/devices/system/node/node%d/cpulist' % node) as f:
            cpus = set()
            for part in f.read().strip().split(','):
                a, _, b = part.partition('-')
                cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
            info.update(bound=True, cpus=len(allowed))
    except Exception as e:        # no NVML / sysfs: run unbound
        info['error'] = repr(e)[:120]
    return info


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU with NVML while the timed region runs."""

    def __init__(self, index, period=0.005):
        threading.Thread.__init__(self, daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            try:
                self.h = pynvml.nvmlDeviceGetHandleByPciBusId(pci_bus_id(index).encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {}
        for nm in ('HwSlowdown', 'HwThermalSlowdown', 'SwThermalSlowdown', 'SwPowerCap', 'HwPowerBrakeSlowdown'):
            for prefix in ('nvmlClocksEventReason', 'nvmlClocksThrottleReason'):
                v = getattr(nv, prefix + nm, None)
                if v is not None:
                    names[nm] = v
                    break
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for nm, bit in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        to_snake = {'HwSlowdown': 'hw_slowdown', 'HwThermalSlowdown': 'hw_thermal_slowdown',
                    'SwThermalSlowdown': 'sw_thermal_slowdown', 'SwPowerCap': 'sw_power_cap',
                    'HwPowerBrakeSlowdown': 'hw_power_brake_slowdown'}
        return {'sm_mhz': float(np.median(self.samples)) if self.samples else None,
                'sm_max_mhz': float(self.max_mhz) if self.max_mhz else None,
                'reasons': sorted(to_snake[r] for r in self.reasons), 'samples': len(self.samples)}


# --------------------------------------------------------------------------------------- CPU side
def usable_cpus():
    import oracle
    usable = oracle.num_cores()
    if hasattr(os, 'sched_getaffinity'):
        usable = min(usable, len(os.sched_getaffinity(0)))
    try:
        with open('/sys/fs/cgroup/cpu.max') as f:
            quota, period = f.read().split()[:2]
        if quota != 'max':
            usable = max(1, min(usable, int(-(-int(quota) // int(period)))))
    except Exception:
        pass
    return usable


def host_info():
    host = {'os_cpu_count': os.cpu_count(),
            'affinity': len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else None}
    try:
        with open('/sys/fs/cgroup/cpu.max') as f:
            host['cgroup_cpu_max'] = f.read().strip()          # "max 100000" = no quota
    except Exception:
        host['cgroup_cpu_max'] = None
    return host


def cpu_port_rate(workload, seconds_target, steps=None, warmup=0, threads=0):
    """Times the oracle C port (the reference algorithm restated, -O2, no FMA) on the host cores with the benchmark
    policy: OS threads over envs (the reference itself is single-threaded numba).  A faster stand-in for the reference
    (1.45x the numba path in the build container), reported beside the real thing."""
    import oracle
    from f1tenth_gym_b200 import maps
    w = WORKLOADS[workload]
    A, B = w['num_agents'], w['num_beams']
    nthreads = threads if threads > 0 else usable_cpus()
    E = max(nthreads, min(w['num_envs'], 256 * nthreads // A))
    omap = oracle.OracleMap.from_yaml(maps.resolve_map_path('example_map'), '.png')
    sims = [oracle.OracleSim(omap, num_agents=A, num_beams=B) for _ in range(E)]
    wp = maps.load_waypoints()
    rng = np.random.default_rng(SEED)
    for s in sims:
        k = int(rng.integers(0, wp.shape[0]))
        s.reset(np.stack([wp[(k - POSE_GAP * i) % wp.shape[0]] for i in range(A)]))
    oracle.rollout(sims, 20, wp, POSE_GAP, SEED, nthreads)       # settle: mixed speeds, some resets
    if steps is None:
        t0 = time.perf_counter()
        oracle.rollout(sims, 2, wp, POSE_GAP, SEED + 1, nthreads)
        per_tick = (time.perf_counter() - t0) / 2
        steps = max(3, int(seconds_target / max(per_tick, 1e-6)))
    if warmup > 0:
        oracle.rollout(sims, warmup, wp, POSE_GAP, SEED + 100, nthreads)
    # one call for all timed ticks: the worker threads are created once and every env advances `steps` ticks on its
    # own (envs never interact), which is the CPU's best case
    t0 = time.perf_counter()
    total, nlook = oracle.rollout(sims, steps, wp, POSE_GAP, SEED + 1000, nthreads)
    dt = time.perf_counter() - t0
    return {'value': total / dt, 'unit': UNIT, 'cores': nthreads, 'kind': 'port',
            'sample': '%d of the workload\'s %d envs x %d agents x %d ticks (%.1f s), oracle C port of the '
                      'reference numba path, %d threads, noise off, same action/auto-reset policy'
                      % (E, w['num_envs'], A, steps, dt, nthreads),
            'seconds': dt, 'steps': steps, 'ms_per_step': 1e3 * dt / steps, 'envs': E,
            'lookups_per_agent_step': nlook / max(total, 1)}


def cpu_reference_rate(workload, steps, warmup, target_step_s=None):
    """The UNMODIFIED reference (numba Simulator.step from oracle/_ref or /root/reference), one process per usable
    core (SURVEY 8d).  None if the reference modules are not available."""
    from oracle import ref_runner
    w = WORKLOADS[workload]
    if w['num_beams'] != 1080 or not ref_runner.available():
        return None       # the reference Simulator has no beam-count parameter (base_classes.py:493-496)
    r = ref_runner.run(w['num_agents'], steps, warmup, target_step_s=target_step_s)
    r.update(unit=UNIT, cores=r['procs'], kind='reference',
             sample='%d processes x %d reference Simulators x %d ticks per step x %d steps (%.1f s): the unmodified numba '
                    'path (base_classes.Simulator.step), %d agents/env, noise off, same action/auto-reset policy'
                    % (r['procs'], r['envs_per_proc'], r['ticks_per_step'], steps, r['seconds'], w['num_agents']))
    return r


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    world = int(os.environ.get('WORLD_SIZE', '1'))
    ref = None
    try:
        ref = cpu_reference_rate(args.workload, args.steps, args.warmup)
    except Exception as e:       # numba missing / broken on this host: fall back to the C port, say so
        sys.stderr.write('reference arm: numba reference unavailable (%r); timing the oracle C port\n' % (e,))
    port = cpu_port_rate(args.workload, 6.0 if ref is not None else None,
                         steps=None if ref is not None else args.steps, warmup=0 if ref is not None else args.warmup)
    r = ref if ref is not None else port
    cpu = {'value': r['value'], 'unit': UNIT, 'cores': r['cores'], 'kind': r['kind'], 'sample': r['sample'],
           'host': host_info(), 'port_value': port['value'], 'port_cores': port['cores'], 'port_sample': port['sample']}
    line = {'impl': 'reference', 'metric': METRIC, 'value': r['value'], 'unit': UNIT, 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': r['ms_per_step'],
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': config_dict(args.workload, max(world, args.gpus)),
            'cpu_baseline': cpu,
            'e2e': {'value': r['value'], 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0,
            'note': 'kind "reference" = the unmodified f1tenth_gym numba path (oracle/_ref, copied by oracle/make_ref.py), one '
                    'process per usable host core; kind "port" = the C restatement (oracle/f110_oracle.c, bit-exact vs the '
                    'numba path on the golden trajectories) when numba cannot run; port_value is always reported'}
    print(json.dumps(line))


# --------------------------------------------------------------------------------------- GPU side
def dump_outputs(sim, out_dir, torch):
    """Writes the observation the last tick handed its caller (what f110_step_host copies out: scans, state, collisions,
    done, lap times and counts) as out_dir/<name>.npy in float32 / float64, so that two builds can be compared output for
    output.  When the scan block is larger than DUMP_SCAN_BYTES, a fixed seeded sample of agent rows stands for it."""
    os.makedirs(out_dir, exist_ok=True)
    NA, B = sim.scans.shape
    n = min(NA, DUMP_SCAN_BYTES // (4 * B))
    rows = np.arange(NA) if n == NA else np.sort(np.random.default_rng(DUMP_SEED).choice(NA, n, replace=False))
    arrays = {'scans_sample': sim.scans[torch.from_numpy(rows).to(sim.device)],
              'state': sim.state, 'collisions': sim.collisions, 'done': sim.done.to(torch.float32),
              'lap_times': sim.lap_times, 'lap_counts': sim.lap_counts}
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + '.npy'), v.cpu().numpy())


def measure_workload(name, K, W, world, rank, dev, dmap, Ke, prof_ticks, f110, torch, dist, reduce_max_scalar,
                     sampler_index=None, packed=False, dump_dir=None):
    """One workload on this rank's GPU -> dict(value, ms_per_step, e2e, roofline, clocks, ...) (whole-job figures)."""
    w = WORKLOADS[name]
    N, A, B = w['num_envs'], w['num_agents'], w['num_beams']
    NA = N * A
    sim = f110.Simulator(f110.maps.DEFAULT_PARAMS, A, SEED + rank, num_envs=N, num_beams=B, device=dev,
                         march_item_beams=int(os.environ.get('F110_MARCH_ITEM_BEAMS', '32')))
    sim.set_device_map(dmap)
    wp_np = f110.maps.load_waypoints()
    wp = torch.from_numpy(wp_np).to(dev)
    # initial poses keyed by GLOBAL env id so that the population does not depend on the GPU count
    ks = np.array([np.random.default_rng(SEED + rank * N + e).integers(0, wp_np.shape[0]) for e in range(N)])
    poses = np.stack([wp_np[(ks - POSE_GAP * i) % wp_np.shape[0]] for i in range(A)], axis=1)
    sim.env_reset(poses)

    gen = torch.Generator(device=dev)
    gen.manual_seed(SEED + 7919 * rank)
    P = min(K + W, 256)

    def make_actions(n):
        u = torch.rand((n, NA, 2), generator=gen, device=dev, dtype=torch.float64)
        u[..., 0] = -0.4189 + 0.8378 * u[..., 0]      # steer ~ U[-0.4189, 0.4189]
        u[..., 1] = 8.0 * u[..., 1]                   # speed ~ U[0, 8]
        return u.contiguous()
    pool = make_actions(P)
    abuf = torch.zeros((NA, 2), dtype=torch.float64, device=dev)
    sim.capture_graph(abuf, autoreset_poses=wp, pose_gap=POSE_GAP, autoreset_seed=SEED + rank, env_level=True)

    flush = torch.empty(FLUSH_BYTES, dtype=torch.uint8, device=dev)
    for t in range(W):
        abuf.copy_(pool[t % P])
        sim.replay()
    torch.cuda.synchronize(dev)

    ev0 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    ev1 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    sampler = ClockSampler(sampler_index) if sampler_index is not None else None
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    if sampler:
        sampler.start()
    wall0 = time.perf_counter()
    for t in range(K):
        flush.zero_()                                 # evict L2 between timed steps (outside the event pair)
        abuf.copy_(pool[(W + t) % P])
        ev0[t].record()
        sim.replay()
        ev1[t].record()
    torch.cuda.synchronize(dev)
    wall = time.perf_counter() - wall0
    clocks = sampler.stop() if sampler else None
    if world > 1:
        dist.barrier()
    if dump_dir is not None:
        dump_outputs(sim, dump_dir, torch)
    step_ms = np.array([a.elapsed_time(b) for a, b in zip(ev0, ev1)])
    dev_ms_total = reduce_max_scalar(float(step_ms.sum()), dev)
    value = K * NA * world / (dev_ms_total * 1e-3)

    # ---- roofline of the dominant kernel (the ray march): CUDA events around it, live, on its stream
    kms = np.zeros(3)
    for t in range(prof_ticks):
        flush.zero_()
        d = sim.step_profile(pool[t % P].view(N, A, 2))
        sim.env_post_step()
        sim.autoreset(wp, POSE_GAP, SEED + rank)
        kms += np.array(d)
    kms /= prof_ticks
    counter = torch.zeros((1,), dtype=torch.int64, device=dev)
    sim.c.lookup_counter = counter.data_ptr()
    for t in range(prof_ticks):
        sim.step(pool[(t + prof_ticks) % P].view(N, A, 2))
        sim.env_post_step()
        sim.autoreset(wp, POSE_GAP, SEED + rank)
    torch.cuda.synchronize(dev)
    sim.c.lookup_counter = None
    L = counter.item() / float(prof_ticks * NA)                 # DT lookups per agent-step, this pose distribution
    bytes_per_agent_step = 8.0 * L + 4.0 * B + 144.0            # fp64 DT element, fp32 range out, state/action/FIFO
    bytes_per_launch = bytes_per_agent_step * NA
    peak, peak_src = measured_peak()
    achieved = bytes_per_launch / (kms[1] * 1e-3) / 1e9
    roofline = {'bound': 'hbm', 'kernel': 'k_march_lean', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
                'frac': achieved / peak, 'traffic': ncu_traffic(name), 'peak_source': peak_src,
                'algorithmic_bytes_per_agent_step': bytes_per_agent_step, 'lookups_per_agent_step': L,
                'bytes_formula': '8*L + 4*B + 144 (fp64 DT element, fp32 range out); survey 4-byte-element variant: frac_4byte',
                'frac_4byte': (4.0 * L + 4.0 * B + 144.0) * NA / (kms[1] * 1e-3) / 1e9 / peak,
                'kernel_ms': {'k_dynamics': kms[0], 'k_march': kms[1], 'k_tail': kms[2]},
                'march_share_of_step': kms[1] / max(kms.sum(), 1e-12),
                'note': 'the 20.5 MB DT table is L2/L1-resident, so real DRAM traffic is far below the '
                        'algorithmic bytes; see profiles/ for ncu DRAM and L2 throughput'}

    # ---- end to end through the host-buffer API (pipelined: the D2H of tick t overlaps the compute of tick t+1)
    # the caller's actions live in host memory; they are written into the pinned action buffer with a plain
    # single-threaded numpy copy (a torch CPU copy_ of > 32 K elements forks an OpenMP team: milliseconds on a 128-thread box)
    host_pool = pool[:min(P, 32)].cpu().numpy()
    sets = sim.make_host_pipeline(depth=2)
    for io in sets:
        io['_actions_np'] = io['actions'].numpy()

    def e2e_loop(n):
        for t in range(n):
            io = sets[t % 2]
            sim.wait_host(io)                                      # obs of tick t-2 is on the host: io is reusable
            np.copyto(io['_actions_np'], host_pool[t % host_pool.shape[0]])   # the caller's new actions (host -> pinned)
            sim.step_host_async(io)
            sim.autoreset(wp, POSE_GAP, SEED + rank)
        for io in sets:
            sim.wait_host(io)
    e2e_loop(6)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    e2e_loop(Ke)
    torch.cuda.synchronize(dev)
    e2e_s = reduce_max_scalar(time.perf_counter() - t0, dev)
    h2d = NA * 2 * 8
    d2h = NA * B * 4 + NA * 7 * 8 + NA * 8 + N + 2 * NA * 8
    e2e = {'value': Ke * NA * world / e2e_s, 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
           'steps': Ke, 'ms_per_step': 1e3 * e2e_s / Ke, 'd2h_gbs_per_gpu': d2h / (e2e_s / Ke) / 1e9,
           'api': 'Simulator.step_host_async -> C ABI f110_step_host_async: per tick pinned H2D of the actions, tick, '
                  'D2H of scans+state+collisions+done+laps into pinned host buffers (2-deep pipeline, the host waits for '
                  'obs t-2 before issuing tick t)'}
    # ---- the same pipeline with the OPT-IN narrow scan block (24-bit fixed point, 3 bytes per beam): reported beside the
    # fp32 figure above, never instead of it
    e2e_u24 = None
    if packed:
        del sets
        sets = sim.make_host_pipeline(depth=2, packed_scans=True)
        for io in sets:
            io['_actions_np'] = io['actions'].numpy()
        e2e_loop(6)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        e2e_loop(Ke)
        torch.cuda.synchronize(dev)
        p_s = reduce_max_scalar(time.perf_counter() - t0, dev)
        d2h_p = NA * B * 3 + NA * 7 * 8 + NA * 8 + N + 2 * NA * 8
        e2e_u24 = {'value': Ke * NA * world / p_s, 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h_p,
                   'steps': Ke, 'ms_per_step': 1e3 * p_s / Ke, 'd2h_gbs_per_gpu': d2h_p / (p_s / Ke) / 1e9,
                   'what': 'opt-in narrow observation: ranges as 24-bit fixed point (2^-19 m steps, |error| <= 9.6e-7 m), packed on the '
                           'device by f110_pack_scans_u24 inside f110_step_host_async; everything else as in e2e'}
    del sets, sim, flush
    torch.cuda.empty_cache()
    return {'value': value, 'e2e_packed_u24': e2e_u24, 'ms_per_step': dev_ms_total / K, 'steps': K, 'warmup': W, 'e2e': e2e, 'roofline': roofline,
            'clocks': clocks, 'wall_ms_per_step_incl_flush': 1e3 * wall / K, 'num_envs_per_gpu': N, 'num_agents': A,
            'num_beams': B,
            'step_ms_percentiles': {'p5': float(np.percentile(step_ms, 5)), 'p50': float(np.percentile(step_ms, 50)),
                                    'p95': float(np.percentile(step_ms, 95))}}


def run_b200(args):
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    import torch
    import torch.distributed as dist
    numa = numa_bind(local_rank)            # before anything pinned is allocated (make_host_pipeline)
    import f1tenth_gym_b200 as f110
    from f1tenth_gym_b200.distributed import reduce_max_scalar, all_gather_obs

    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        # NCCL prints its version banner to stdout while the communicator is created (NCCL_DEBUG=VERSION ignores
        # NCCL_DEBUG_FILE); stdout must carry exactly one JSON line, so fd 1 points at stderr during the set-up
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group('nccl', rank=rank, world_size=world,
                                    device_id=torch.device('cuda', local_rank))
            torch.cuda.set_device(local_rank)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    K, W = args.steps, args.warmup
    dmap = f110.DeviceMap.from_yaml(f110.maps.resolve_map_path('example_map'), '.png', dev)
    common = dict(world=world, rank=rank, dev=dev, dmap=dmap, f110=f110, torch=torch, dist=dist,
                  reduce_max_scalar=reduce_max_scalar)
    main = measure_workload(args.workload, K, W, Ke=min(K, 200), prof_ticks=20, sampler_index=local_rank, packed=True,
                            dump_dir=args.dump_outputs if rank == 0 else None, **common)

    # optional NCCL observation all-gather for a single-process trainer (SURVEY 8e), timed OFF the step path
    gather = None
    if world > 1:
        w = WORKLOADS[args.workload]
        shard = torch.zeros((w['num_envs'] * w['num_agents'], w['num_beams']), dtype=torch.float32, device=dev)
        sizes = [shard.shape[0]] * world              # equal shards: one all_gather_into_tensor, no size exchange
        full = torch.empty((shard.shape[0] * world, shard.shape[1]), dtype=shard.dtype, device=dev)
        for _ in range(3):
            all_gather_obs(shard, sizes=sizes, out=full)
        torch.cuda.synchronize(dev)
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 10
        e0.record()
        for _ in range(reps):
            all_gather_obs(shard, sizes=sizes, out=full)
        e1.record()
        torch.cuda.synchronize(dev)
        ms = reduce_max_scalar(e0.elapsed_time(e1) / reps, dev)
        recv = shard.numel() * 4 * (world - 1)
        gather = {'ms': ms, 'shard_bytes': shard.numel() * 4, 'gathered_bytes': full.numel() * 4,
                  'recv_gbs_per_gpu': recv / (ms * 1e-3) / 1e9,
                  'what': 'distributed.all_gather_obs (NCCL all_gather over NVLink) of the fp32 scan shard of every rank, '
                          'off the step path, CUDA events, max over ranks'}
        del shard, full
        torch.cuda.empty_cache()

    extras = {}
    if world == 1 and not args.no_extras:
        for name in EXTRA_WORKLOADS:
            if name == args.workload:
                continue
            r = measure_workload(name, min(K, 100), min(max(W, 3), 10), Ke=120, prof_ticks=8, **common)
            extras[name] = {k: r[k] for k in ('value', 'ms_per_step', 'steps', 'warmup', 'e2e', 'roofline', 'num_envs_per_gpu',
                                              'num_agents', 'num_beams')}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        port = cpu_port_rate(args.workload, args.cpu_seconds)
        ref = None
        try:
            ref = cpu_reference_rate(args.workload, steps=10, warmup=2, target_step_s=1.0)
        except Exception as e:
            sys.stderr.write('cpu_baseline: numba reference unavailable (%r); reporting the C port\n' % (e,))
        r = ref if ref is not None else port
        cpu = {'value': r['value'], 'unit': UNIT, 'cores': r['cores'], 'kind': r['kind'], 'sample': r['sample'],
               'host': host_info(), 'port_value': port['value'], 'port_cores': port['cores'], 'port_sample': port['sample'],
               'lookups_per_agent_step': port['lookups_per_agent_step']}

    if rank == 0:
        cfg = config_dict(args.workload, world)
        line = {'metric': METRIC, 'value': main['value'], 'unit': UNIT, 'n_gpus': world, 'steps': K, 'warmup': W,
                'ms_per_step': main['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': 'f64', 'data': 'synthetic', 'config': cfg,
                'measurement': {'actions': 'pregenerated in HBM', 'auto_reset': 'in the timed tick (hashed start pose)',
                                'l2': 'flushed between timed steps (256 MiB memset outside the per-step CUDA-event pairs)',
                                'timing': 'sum of per-step CUDA-event times on the launch stream, max over ranks',
                                'numa': numa},
                'clocks': main['clocks'], 'e2e': main['e2e'], 'e2e_packed_u24': main['e2e_packed_u24'],
                # per tick: k_dynamics (+ march queue build), k_march_lean, k_tail (finalize + lap logic + auto-reset)
                'gpu_launches': 3 * K, 'roofline': main['roofline'], 'cpu_baseline': cpu,
                'wall_ms_per_step_incl_flush': main['wall_ms_per_step_incl_flush'],
                'step_ms_percentiles': main['step_ms_percentiles'], 'workloads': extras}
        if gather is not None:
            line['obs_all_gather'] = gather
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=500)
    ap.add_argument('--warmup', type=int, default=50)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument('--cpu-seconds', type=float, default=10.0)
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-extras', action='store_true', help='skip the other BASELINE configs (1 GPU only)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write the observation of the last one (rank 0) as DIR/<name>.npy')
    args = ap.parse_args()
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs needs --impl b200')
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
