"""f1tenth_gym_b200 — B200-native batched F1TENTH simulator hot path.

Drop-in for the per-tick path of f1tenth/f1tenth_gym (Simulator.step: pid + RK4 single-track dynamics,
1080-beam lidar ray-march on the distance-transform grid, iTTC, opponent ray-cast, GJK collision)
behind the reference's own Python surface (F110Env / Simulator / ScanSimulator2D and the @njit kernel
names).  Compute happens only in libf110_b200.so (hand-written sm_100a CUDA behind a C ABI).
"""
from .simulator import Integrator, Simulator, DeviceMap, DeviceBeams   # noqa: F401
from .env import F110Env                                              # noqa: F401
from . import kernels, maps, trackgen                                 # noqa: F401
from .kernels import ScanSimulator2D                                  # noqa: F401
from .planner import PurePursuitPlanner                               # noqa: F401
from .render import RenderView                                        # noqa: F401

__all__ = ['F110Env', 'Simulator', 'Integrator', 'ScanSimulator2D', 'PurePursuitPlanner', 'DeviceMap', 'DeviceBeams', 'RenderView',
           'kernels', 'maps', 'trackgen']
