// f110_b200.cu — kernels and C ABI of libf110_b200.so (see include/f110_b200.h).
//
// One tick (reference base_classes.py:553-612 Simulator.step) = three launches on the caller's stream:
//   k_dynamics     thread per agent     steer FIFO, pid, RK4/Euler, yaw wrap, scan pose, pose snapshot, the per-agent record of
//                                       the march (+ extra blocks that sort last tick's work items into the march queue)
//   k_march_lean   persistent, warp per 32-beam item (march_lean.cuh): LUT heading, sphere tracing on the DT grid, fused iTTC
//                                       predicate, optional seeded noise, fp32 range out -- the roofline kernel.  Maps with a
//                                       rotated origin and stand-alone scans run the literal k_raymarch (thread per beam)
//   k_tail         warp per agent       GJK vs. the other agents of the env, wall-hit state zeroing, opponent ray-cast inside the
//                                       blocked-view window, collisions obs, then lap logic and auto-reset per env
//                                       (k_finalize = the same without the env-level part, for f110_step)
// Off the tick path, f110_render draws top-down frames of the state (render.cuh): k_render_frame (4 pixels per thread), then the
// scan-endpoint and waypoint layers as stream-ordered scatter launches.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -fmad=false (no FMA contraction).
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>

#include "../../include/f110_b200.h"
#include "collision.cuh"
#include "dynamics.cuh"
#include "lidar.cuh"
#include "march.cuh"
#include "march_lean.cuh"
#include "march_tile.cuh"
#include "planner.cuh"
#include "edt.cuh"
#include "trackgen.cuh"
#include "render.cuh"

namespace f110 {

static thread_local char g_cuda_err[256] = "";

static int cuda_fail(cudaError_t e, const char *where) {
    snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s", where, cudaGetErrorString(e));
    return F110_ERR_CUDA;
}
#define CUDA_TRY(call)                                                   \
    do {                                                                 \
        cudaError_t e__ = (call);                                        \
        if (e__ != cudaSuccess) return cuda_fail(e__, #call);            \
    } while (0)
#define LAUNCH_CHECK(name)                                               \
    do {                                                                 \
        cudaError_t e__ = cudaGetLastError();                            \
        if (e__ != cudaSuccess) return cuda_fail(e__, name);             \
    } while (0)

static MapView make_view(const f110_map *m) {
    MapView v;
    v.dt = m->dt; v.dt_cells = m->dt_cells; v.dt_codes = m->dt_codes; v.dt_lut = m->dt_lut;
    v.sines = m->sines; v.cosines = m->cosines;
    v.orig_x = m->orig_x; v.orig_y = m->orig_y; v.orig_c = m->orig_c; v.orig_s = m->orig_s;
    v.resolution = m->resolution; v.inv_resolution = 1.0 / m->resolution;
    v.x_max = m->width * m->resolution;    // `width * resolution` (laser_models.py:79)
    v.y_max = m->height * m->resolution;
    v.eps = m->eps; v.max_range = m->max_range; v.dt_oob = m->dt_oob;
    v.theta_dis = m->theta_dis; v.theta_dis_f = (double)m->theta_dis;
    v.height = m->height; v.width = m->width;
    return v;
}

struct BeamView {
    const double *__restrict__ scan_angles;
    const double *__restrict__ cosines;
    const double *__restrict__ side_distances;
    double fov, angle_increment, theta_index_increment;
    int32_t num_beams;
};
static BeamView make_view(const f110_beams *b) {
    BeamView v;
    v.scan_angles = b->scan_angles; v.cosines = b->cosines; v.side_distances = b->side_distances;
    v.fov = b->fov; v.angle_increment = b->angle_increment; v.theta_index_increment = b->theta_index_increment;
    v.num_beams = b->num_beams;
    return v;
}

// Work queue of the persistent march kernel (march.cuh): sort the 32-beam items into [very heavy | heavy |
// light] by the maximum lookup count they recorded in the previous tick.  One thread per item; runs as the
// extra blocks of k_dynamics (it only reads march_cost, which the reset kernels mark as unknown).
#define F110_ORDER_ITEMS_PER_THREAD 8
__device__ __forceinline__ void build_march_order(const f110_sim &s, unsigned first_block, unsigned items) {
    // Round 2 (profiles/r2/dynamics_cfg3_line_hot.txt: the builder was 65 % of k_dynamics' instructions at cfg3 -- 24 ballots
    // and up to 24 shared atomics per thread, a runtime division per item): a thread owns EIGHT CONSECUTIVE items, so
    //   * one division per thread (the items after the first step (agent, slice) incrementally),
    //   * the neighbours of an item are the thread's own registers (only the two ends are extra loads: 10 loads, not 24),
    //   * the per-class counts of a thread are packed into one word (3 x 10 bits) and ONE warp scan places all of them,
    //   * a warp touches the three shared counters once, the block the three global ones once,
    // and a class list is in item order within a block, i.e. consecutive entries are neighbouring slices of one agent.
    __shared__ unsigned s_cnt[3], s_base[3];
    const unsigned lane = threadIdx.x & 31u;
    const unsigned ipa = (unsigned)s.march_ipa;
    if (threadIdx.x < 3) s_cnt[threadIdx.x] = 0u;
    const unsigned t = (blockIdx.x - first_block) * blockDim.x + threadIdx.x;
    const unsigned w0 = t * F110_ORDER_ITEMS_PER_THREAD;
    unsigned packed[F110_ORDER_ITEMS_PER_THREAD], c[F110_ORDER_ITEMS_PER_THREAD + 2];
    int cls[F110_ORDER_ITEMS_PER_THREAD];
    unsigned a = 0, j = 0;
    if (w0 < items) { a = w0 / ipa; j = w0 - a * ipa; }
    // c[0] = left neighbour of the first item, c[1..8] = the items, c[9] = right neighbour of the last one
    c[0] = (w0 < items && j > 0) ? s.march_cost[((a << 8) | j) - 1u] : F110_Q_UNKNOWN;
    unsigned aa = a, jj = j;
#pragma unroll
    for (int k = 0; k < F110_ORDER_ITEMS_PER_THREAD; k++) {
        const bool live = w0 + (unsigned)k < items;
        packed[k] = (aa << 8) | jj;
        c[k + 1] = live ? s.march_cost[packed[k]] : F110_Q_UNKNOWN;
        cls[k] = live ? 0 : -1;
        if (++jj == ipa) { jj = 0; aa++; }
    }
    {
        const unsigned wl = w0 + F110_ORDER_ITEMS_PER_THREAD;      // the item after this thread's last one
        c[F110_ORDER_ITEMS_PER_THREAD + 1] = (wl < items && jj > 0) ? s.march_cost[(aa << 8) | jj] : F110_Q_UNKNOWN;
    }
    unsigned mine = 0u;                                             // per-class counts, 10 bits each
#pragma unroll
    for (int k = 0; k < F110_ORDER_ITEMS_PER_THREAD; k++) {
        if (cls[k] == 0) {
            const unsigned sj = packed[k] & 255u;
            unsigned m = c[k + 1];
            if (m != F110_Q_UNKNOWN) {
                // neighbours only inside the same agent: slice 0 has no left one, slice ipa-1 no right one
                if (sj > 0 && c[k] != F110_Q_UNKNOWN) m = max(m, c[k]);
                if (sj + 1 < ipa && c[k + 2] != F110_Q_UNKNOWN) m = max(m, c[k + 2]);
            }
            cls[k] = (c[k + 1] == F110_Q_UNKNOWN || c[k + 1] >= F110_Q_VERY_HEAVY) ? 0 : (m >= F110_Q_HEAVY) ? 1 : 2;
            mine += 1u << (10 * cls[k]);
        }
    }
    // exclusive warp scan of the packed counts (a warp holds at most 256 items per class: 9 bits)
    unsigned incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned v = __shfl_up_sync(0xffffffffu, incl, o);
        if ((int)lane >= o) incl += v;
    }
    const unsigned excl = incl - mine;
    const unsigned wtot = __shfl_sync(0xffffffffu, incl, 31);
    __syncthreads();                                                // s_cnt zeroed
    unsigned wbase = 0u;                                            // lanes 0..2 fetch the warp's base of class `lane`
    if (lane < 3u) {
        const unsigned n = (wtot >> (10 * lane)) & 1023u;
        wbase = n ? atomicAdd(&s_cnt[lane], n) : 0u;
    }
    const unsigned b0 = __shfl_sync(0xffffffffu, wbase, 0), b1 = __shfl_sync(0xffffffffu, wbase, 1),
                   b2 = __shfl_sync(0xffffffffu, wbase, 2);
    __syncthreads();
    if (threadIdx.x < 3) s_base[threadIdx.x] = s_cnt[threadIdx.x] ? atomicAdd(s.march_count + threadIdx.x, s_cnt[threadIdx.x]) : 0u;
    __syncthreads();
    unsigned pos[3] = { s_base[0] + b0 + (excl & 1023u), s_base[1] + b1 + ((excl >> 10) & 1023u),
                        s_base[2] + b2 + ((excl >> 20) & 1023u) };
#pragma unroll
    for (int k = 0; k < F110_ORDER_ITEMS_PER_THREAD; k++) {
        if (cls[k] >= 0) {
            const unsigned at = (cls[k] == 0) ? pos[0]++ : (cls[k] == 1) ? pos[1]++ : pos[2]++;
            if (at < items) s.march_order[(size_t)cls[k] * items + at] = packed[k];
        }
    }
}

// Agent-level queue of the tile march kernel (march_tile.cuh): one thread per agent classifies it by the largest
// per-slice lookup maximum of the previous tick (unknown = very heavy), same three classes, lists in march_order[3][M].
__device__ __forceinline__ void build_agent_order(const f110_sim &s, unsigned first_block, unsigned agents) {
    __shared__ unsigned s_cnt[3], s_base[3];
    if (threadIdx.x < 3) s_cnt[threadIdx.x] = 0u;
    __syncthreads();
    const unsigned a = (blockIdx.x - first_block) * blockDim.x + threadIdx.x;
    int cls = -1;
    unsigned slot = 0;
    if (a < agents) {
        unsigned m = 0;
        for (int j = 0; j < s.march_ipa; j++) m = max(m, s.march_cost[((size_t)a << 8) + (size_t)j]);     // unknown = 0xFFFFFFFF wins
        cls = (m >= F110_Q_VERY_HEAVY) ? 0 : (m >= F110_Q_HEAVY) ? 1 : 2;
        slot = atomicAdd(&s_cnt[cls], 1u);
    }
    __syncthreads();
    if (threadIdx.x < 3) s_base[threadIdx.x] = s_cnt[threadIdx.x] ? atomicAdd(s.march_count + threadIdx.x, s_cnt[threadIdx.x]) : 0u;
    __syncthreads();
    if (cls >= 0) {
        const unsigned at = s_base[cls] + slot;
        if (at < agents) s.march_order[(size_t)cls * agents + at] = a;
    }
}

// ------------------------------------------------------------------------------------ k_dynamics
struct FirstLookup {
    const double *__restrict__ cells;    // dt / res (cell units) or dt (metres), or NULL: generic march kernel
    double ox, oy, inv_res;              // cell units
    double res, orig_x, orig_y, x_max, y_max;   // metres
    unsigned width, height, last;
    int metres;
    const int32_t *__restrict__ env_layer;   // multi-map batches: layer of each env, or NULL
    unsigned long long layer_stride;
    // per-agent record of the lean march kernel (march_lean.cuh); rec == NULL: not written
    double2 *__restrict__ rec;
    double side_max, ttc_margin;
    unsigned long long rec_layer_stride;     // elements between map layers of the table the lean kernel reads
    int agent_queue;                         // 1: the extra blocks build the agent-level queue of the tile march kernel
};

__global__ void __launch_bounds__(128) k_dynamics(f110_sim s, const double *__restrict__ actions, double fov,
                                                  double theta_dis_f, int dyn_blocks, FirstLookup fl) {
    const int NA = s.num_envs * s.num_agents;
    pdl_launch_dependents();                 // the march kernel may start its launch / prologue now (it waits before reading)
    if ((int)blockIdx.x >= dyn_blocks) {     // extra blocks: build the march work queue (block-uniform branch)
        if (fl.agent_queue) build_agent_order(s, (unsigned)dyn_blocks, (unsigned)NA);
        else build_march_order(s, (unsigned)dyn_blocks, (unsigned)NA * (unsigned)s.march_ipa);
        return;
    }
    const int a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= NA) return;
    // the tick counter advances once per tick, here, before any kernel of the tick reads it (noise stream id,
    // auto-reset draw); nothing else in this kernel uses it
    if (a == 0 && s.tick_counter) *s.tick_counter += 1ull;
    const double *p = s.params + (size_t)(s.params_per_env ? a : a % s.num_agents) * F110_NPARAM;
    double st[7];
#pragma unroll
    for (int k = 0; k < 7; k++) st[k] = s.state[(size_t)k * NA + a];
    // steering delay FIFO (base_classes.py:270-278): depth 2, zeros until two commands are queued
    const double raw_steer = actions[2 * (size_t)a], speed = actions[2 * (size_t)a + 1];
    int cnt = s.steer_cnt[a];
    double b0 = s.steer_buf[a], b1 = s.steer_buf[(size_t)NA + a];
    double steer = (cnt < 2) ? 0. : b1;
    s.steer_buf[(size_t)NA + a] = b0;
    s.steer_buf[a] = raw_steer;
    if (cnt < 2) s.steer_cnt[a] = cnt + 1;

    integrate_tick(st, steer, speed, p, s.timestep, s.integrator);

#pragma unroll
    for (int k = 0; k < 7; k++) s.state[(size_t)k * NA + a] = st[k];
    // scan pose (base_classes.py:406-409) and the first beam's LUT index (laser_models.py:167-172)
    double sx = st[0], sy = st[1];
    if (s.lidar_dist != 0.0) {
        sx = st[0] + s.lidar_dist * cos(st[4]);
        sy = st[1] + s.lidar_dist * sin(st[4]);
    }
    // slot 2: on fast-path maps the DT value of the scan-pose cell in cell units — the first lookup of every
    // beam of this agent (laser_models.py:129), done once here; otherwise the yaw
    double slot2 = st[4];
    const size_t lo = fl.env_layer ? (size_t)fl.env_layer[a / s.num_agents] * (size_t)fl.layer_stride : (size_t)0;
    if (fl.cells && !fl.metres) {
        CellConsts k;
        k.ox = fl.ox; k.oy = fl.oy; k.eps = 0; k.tmax = 0; k.width = fl.width; k.height = fl.height; k.last = fl.last;
        slot2 = __ldg(fl.cells + lo + cell_index(sx * fl.inv_res, sy * fl.inv_res, k));
    } else if (fl.cells) {          // literal xy_2_rc (laser_models.py:55-86), unrotated origin
        const double tx = sx - fl.orig_x, ty = sy - fl.orig_y;
        unsigned idx = fl.last;
        if (!(tx < 0 || tx >= fl.x_max || ty < 0 || ty >= fl.y_max))
            idx = (unsigned)(int)(ty / fl.res) * fl.width + (unsigned)(int)(tx / fl.res);
        slot2 = __ldg(fl.cells + lo + idx);
    }
    double2 *sp = reinterpret_cast<double2 *>(s.scan_pose) + 2 * (size_t)a;
    const double ti0 = theta_index0(st[4], fov, theta_dis_f);
    sp[0] = make_double2(sx, sy);
    sp[1] = make_double2(slot2, ti0);
    if (fl.rec) {
        // everything the march needs per agent, computed once here instead of once per 32-beam work item
        // the march takes floor() through the low word of a magic-number add: cell coordinates must stay below 2^31
        const bool sane = fabs(sx) * fl.inv_res < 1e9 && fabs(sy) * fl.inv_res < 1e9;
        const bool cells = !fl.metres;
        double2 *rp = fl.rec + 4 * (size_t)a;
        rp[0] = (sane && cells) ? make_double2(sx * fl.inv_res, sy * fl.inv_res) : make_double2(sx, sy);
        // LUT index of beam 0 as Q16.48 (ti0 in [0, theta_dis], theta_dis < 2^15); all ones = absurd coordinates
        const unsigned long long tfx = sane ? __double2ull_rd(ti0 * 281474976710656.0) : ~0ull;
        rp[1] = make_double2(slot2, __longlong_as_double((long long)tfx));
        // iTTC (laser_models.py:188-217) can only fire for |range - side_i| <= margin * |v cos_i|, i.e. never for
        // range > max(side) + margin * |v| (1e-9 of slack covers the roundings); v == 0 never fires
        const double v = st[3];
        const double thr = (v != 0.0) ? (fl.side_max + fl.ttc_margin * fabs(v)) * (1.0 + 1e-9) : -INFINITY;
        rp[2] = make_double2(thr, v);
        const unsigned long long lo_rec = fl.env_layer ? (unsigned long long)fl.env_layer[a / s.num_agents] * fl.rec_layer_stride : 0ull;
        rp[3] = make_double2(__longlong_as_double((long long)lo_rec), ti0);
    }
    // pose snapshot (Simulator.agent_poses, base_classes.py:574) + cos/sin of the yaw: every vertex / heading
    // computation of the finalize kernel reuses them instead of re-evaluating fp64 trig per opponent
    double *ap = s.agent_poses + 5 * (size_t)a;
    ap[0] = st[0]; ap[1] = st[1]; ap[2] = st[4];
    sincos(st[4], ap + 4, ap + 3);
    s.wall_flag[a] = 0;
}

// ------------------------------------------------------------------------------------ k_raymarch
// One thread per beam; a warp owns 32 consecutive beams of (mostly) one agent, so its lanes walk
// neighbouring cells of the DT grid.  The grid is read through the read-only path: per scan the
// ~7-8 k lookups touch only ~1.3 k distinct 32-byte sectors (measured, DESIGN.md), i.e. the working
// set of the agents resident on an SM lives in L1 and the whole 20 MB table in L2.
struct MarchArgs {
    const double *__restrict__ scan_pose;   // [M][4] (x, y, yaw, theta_index0)    (STANDALONE: [M][3])
    const double *__restrict__ vel;         // [M] longitudinal velocity for iTTC, or NULL
    float *__restrict__ out_f32;            // [M][B] or NULL
    double *__restrict__ out_f64;           // [M][B] or NULL
    int32_t *__restrict__ wall_flag;        // [M] or NULL
    unsigned long long *lookup_counter;     // [1] or NULL
    const unsigned long long *tick_counter; // [1] or NULL (noise stream id)
    double ttc_thresh, noise_std;
    unsigned long long noise_seed;
    long long total;                        // M * B
};

template <bool FAST, bool STANDALONE>
__global__ void __launch_bounds__(256) k_raymarch(MapView m, BeamView bv, MarchArgs g) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = gid < g.total;
    int nlook = 0;
    if (valid) {
        const int B = bv.num_beams;
        const int a = (int)(gid / B);
        const int i = (int)(gid - (long long)a * B);
        double px, py, ti0;
        if (STANDALONE) {
            px = g.scan_pose[3 * (size_t)a];
            py = g.scan_pose[3 * (size_t)a + 1];
            ti0 = theta_index0(g.scan_pose[3 * (size_t)a + 2], bv.fov, m.theta_dis_f);
        } else {
            const double2 *sp = reinterpret_cast<const double2 *>(g.scan_pose) + 2 * (size_t)a;
            const double2 xy = __ldg(sp), yt = __ldg(sp + 1);
            px = xy.x; py = xy.y; ti0 = yt.y;
        }
        const int ti = beam_theta_index(ti0, i, bv.theta_index_increment, m.theta_dis_f);
        const double s = __ldg(m.sines + ti), c = __ldg(m.cosines + ti);
        double range = trace_ray<FAST>(m, px, py, s, c, nlook);
        if (g.noise_std > 0.0) {
            unsigned long long tick = g.tick_counter ? *g.tick_counter : 0ull;
            range = range + g.noise_std * normal_sample(g.noise_seed, tick, (uint64_t)gid);
        }
        if (g.wall_flag) {
            const double v = __ldg(g.vel + a);
            if (ttc_hit(range, v, __ldg(bv.cosines + i), __ldg(bv.side_distances + i), g.ttc_thresh))
                atomicOr(g.wall_flag + a, 1);
        }
        if (g.out_f32) g.out_f32[gid] = (float)range;
        if (g.out_f64) g.out_f64[gid] = range;
    }
    if (g.lookup_counter) {
        unsigned n = (unsigned)nlook;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
        if ((threadIdx.x & 31) == 0 && n) atomicAdd(g.lookup_counter, (unsigned long long)n);
    }
}

// ------------------------------------------------------------------------------------ finalize
// One warp finalises one agent (base_classes.py:536-550 check_collision, :579-589 update_scan loop).
__device__ __forceinline__ void finalize_agent(const f110_sim &s, const BeamView &bv, int a, int lane,
                                               double max_scan_range) {
    const int NA = s.num_envs * s.num_agents;
    const int A = s.num_agents;
    const int env = a / A, slot = a - env * A;
    const int hit = s.wall_flag[a];
    const double *pa = s.agent_poses + 5 * (size_t)a;
    const double px = pa[0], py = pa[1];      // == state[0], state[1]
    // check_ttc zeroes state[3:] — including the yaw — before the opponent ray-cast reads it (:246-249, :225)
    const double yaw = hit ? 0.0 : pa[2];
    const double cyaw = hit ? 1.0 : pa[3], syaw = hit ? 0.0 : pa[4];
    if (hit && lane < 4) s.state[(size_t)(3 + lane) * NA + a] = 0.0;

    // GJK against the other agents of this env, lower index first (collision_multiple :184-212)
    int col = 0, cidx = -1;
    if (A > 1) {
        double vme[8];
        get_vertices_cs(pa[0], pa[1], pa[3], pa[4], s.sim_length, s.sim_width, vme);
        // two car bodies can only overlap if their centres are closer than one body diagonal; beyond that
        // (with a 0.1 % margin) the shapes are strictly separated and GJK returns False, so it is not run
        const double reach2 = (s.sim_length * s.sim_length + s.sim_width * s.sim_width) * 1.001;
        for (int j = lane; j < A; j += 32) {
            if (j == slot) continue;
            const double *pb = s.agent_poses + 5 * (size_t)(env * A + j);
            const double ddx = pb[0] - pa[0], ddy = pb[1] - pa[1];
            if (ddx * ddx + ddy * ddy > reach2) continue;
            double vo[8];
            get_vertices_cs(pb[0], pb[1], pb[3], pb[4], s.sim_length, s.sim_width, vo);
            bool c = (slot < j) ? gjk_collision(vme, vo) : gjk_collision(vo, vme);
            if (c) { col = 1; cidx = max(cidx, j); }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            col |= __shfl_xor_sync(0xffffffffu, col, o);
            cidx = max(cidx, __shfl_xor_sync(0xffffffffu, cidx, o));
        }
    }
    if (lane == 0) {
        s.collisions[a] = (col || hit) ? 1.0 : 0.0;
        s.collision_idx[a] = cidx;
    }

    // ray_cast_agents (:206-227): opponents in ascending index, each bounded to its blocked-view window
    if (A > 1) {
        const double *p = s.params + (size_t)(s.params_per_env ? a : slot) * F110_NPARAM;
        const double length = p[P_LENGTH], width = p[P_WIDTH];
        float *scan = s.scans + (size_t)a * bv.num_beams;
        // an opponent whose nearest point is farther than any range the scan can hold (max_range plus noise
        // head-room) cannot shorten a beam: ray_cast would leave the scan unchanged, so it is skipped
        const double half_diag = 0.5 * sqrt(length * length + width * width);
        for (int j = 0; j < A; j++) {
            if (j == slot) continue;
            const double *pb = s.agent_poses + 5 * (size_t)(env * A + j);
            {
                const double ddx = pb[0] - px, ddy = pb[1] - py;
                const double far = max_scan_range + half_diag;
                if (ddx * ddx + ddy * ddy > far * far) continue;
            }
            double v[8];
            get_vertices_cs(pb[0], pb[1], pb[3], pb[4], length, width, v);
            int lo, hi;
            double phi;
            blocked_view_indices_warp(px, py, cyaw, syaw, v, bv.scan_angles, bv.num_beams, bv.fov, bv.angle_increment,
                                      lane, pb[0], pb[1], lo, hi, phi);
            // When the opponent straddles the rear cut of the field of view the window is ALL beams
            // (laser_models.py:310-315 takes min/max of the four nearest-beam indices).  A ray can only meet an
            // edge if it points into the cone that contains the opponent's bounding circle, so beams outside
            // that cone (+0.05 rad of slack) would get four `inf` ranges and leave the scan unchanged: skip them.
            // The cone (an asin and a sqrt) is only worth computing for a WIDE window; a narrow window (opponent in front)
            // consists of beams that point at the opponent anyway, so it runs unfiltered (cone = 4 > pi).
            double cone = 4.0;      // > pi: no filtering (also when the ego is inside / next to the bounding circle)
            const bool wide = hi - lo >= 96;
            if (wide) {
                const double ddx = pb[0] - px, ddy = pb[1] - py;
                const double dist = sqrt(ddx * ddx + ddy * ddy);
                if (dist > 1.25 * half_diag) cone = asin(half_diag / dist) + 0.05;
            }
            // one beam of the window: cone test, then the four edges (only `min(scan, range)` is needed)
            auto cast_beams = [&](int i0, int i1) {
                for (int i = i0 + lane; i <= i1; i += 32) {
                    const float cur = scan[i];          // issued early: often an L2/DRAM miss (the march just wrote it)
                    double bt = yaw + bv.scan_angles[i];
                    double dl = bt - phi;
                    dl = dl - (2 * M_PI) * rint(dl * (1.0 / (2 * M_PI)));
                    // (the mirrored cone is kept too: get_range's collinear branch, laser_models.py:275-278, has no
                    // direction test, so a beam pointing exactly away along an edge line still reports that edge)
                    const double adl = fabs(dl);
                    if (adl > cone && (M_PI - adl) > cone) continue;
                    double v3x, v3y;
                    sincos(bt + M_PI / 2., &v3y, &v3x);
                    const double curd = (double)cur;
                    double r = INFINITY;
#pragma unroll
                    for (int e = 0; e < 4; e++) {
                        int e2 = (e + 1) & 3;
                        double d = get_range_below(px, py, v3x, v3y, v[2 * e], v[2 * e + 1], v[2 * e2], v[2 * e2 + 1], curd);
                        if (d < r) r = d;
                    }
                    float rf = (float)r;
                    if (rf < cur) scan[i] = rf;
                }
            };
            if (cone < 3.5 && wide) {
                // wide window (the opponent straddles the rear cut: ALL beams): only beams whose angle lies within `cone` of
                // the direction to the opponent, or of the opposite direction, can pass the test above.  Those are the
                // beams around the centres (phi - yaw) + m pi; visit just these index intervals, with two beams of slack
                // on both sides -- the exact per-beam test still decides.
                const double base = phi - yaw, half = bv.fov / 2., inv_inc = 1.0 / bv.angle_increment;
                // centres base + m pi that can reach the beam range [-half, half] (+- cone and slack): usually 1-3 of them
                const int m0 = max(-3, (int)floor((-half - cone - 0.02 - base) * (1.0 / M_PI))),
                          m1 = min(5, (int)ceil((half + cone + 0.02 - base) * (1.0 / M_PI)));
                for (int m = m0; m <= m1; m++) {
                    const double c = base + (double)m * M_PI;
                    const double f0 = (c - cone + half) * inv_inc - 2.0, f1 = (c + cone + half) * inv_inc + 2.0;
                    if (f1 < (double)lo || f0 > (double)hi) continue;
                    const int i0 = max(lo, (int)floor(fmax(f0, (double)lo))), i1 = min(hi, (int)ceil(fmin(f1, (double)hi)));
                    cast_beams(i0, i1);
                }
            } else {
                cast_beams(lo, hi);
            }
            __syncwarp();
        }
    }
}

// the march work-queue counters are consumed once k_march has run; the next tick's k_dynamics refills them
__device__ __forceinline__ void end_of_tick_housekeeping(const f110_sim &s) {
    if (s.march_count) { s.march_count[0] = 0u; s.march_count[1] = 0u; s.march_count[2] = 0u; s.march_count[3] = 0u; }
}

// f110_step: warp per agent
__global__ void __launch_bounds__(128, 8) k_finalize(f110_sim s, BeamView bv, double max_scan_range) {
    pdl_wait();
    const int a = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (a >= s.num_envs * s.num_agents) return;
    finalize_agent(s, bv, a, lane, max_scan_range);
    if (a == 0 && lane == 0) end_of_tick_housekeeping(s);
}

// ------------------------------------------------------------------------------------ reset kernels
// a reset agent has no lookup history: its march items are scheduled with the very-heavy class next tick
__device__ __forceinline__ void mark_march_cost_unknown(const f110_sim &s, size_t a) {
    if (s.march_cost)
        for (int j = 0; j < s.march_ipa; j++) s.march_cost[(a << 8) + (size_t)j] = F110_Q_UNKNOWN;
}

__global__ void k_reset(f110_sim s, const double *__restrict__ poses, const uint8_t *__restrict__ mask) {
    const int NA = s.num_envs * s.num_agents;
    const int a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= NA) return;
    if (mask && !mask[a / s.num_agents]) return;
    // RaceCar.reset base_classes.py:183-204
#pragma unroll
    for (int k = 0; k < 7; k++) s.state[(size_t)k * NA + a] = 0.0;
    s.state[a] = poses[3 * (size_t)a];
    s.state[(size_t)NA + a] = poses[3 * (size_t)a + 1];
    s.state[(size_t)4 * NA + a] = poses[3 * (size_t)a + 2];
    s.steer_cnt[a] = 0;
    s.steer_buf[a] = 0.0;
    s.steer_buf[(size_t)NA + a] = 0.0;
    s.wall_flag[a] = 0;
    mark_march_cost_unknown(s, a);
}

// clear_done: f110_env_reset (a fresh episode requested by the caller) clears the done flag; the auto-reset does NOT --
// the tick that ended an episode must still report done = 1 for it (the next tick recomputes the flag)
__device__ __forceinline__ void env_counters_reset(const f110_sim &s, int env, const double *agent_pose3 /* [A][3] */,
                                                   bool clear_done = true) {
    const int A = s.num_agents;
    s.current_time[env] = 0.0;
    for (int i = 0; i < A; i++) {
        const size_t a = (size_t)env * A + i;
        s.near_starts[a] = 1;
        s.toggle_list[a] = 0.0;
        s.start_xs[a] = agent_pose3[3 * i];
        s.start_ys[a] = agent_pose3[3 * i + 1];
        s.start_thetas[a] = agent_pose3[3 * i + 2];
    }
    // f110_env.py:331 start_rot from the ego's start heading
    const double th = -agent_pose3[3 * s.ego_idx + 2];
    double *R = s.start_rot + 4 * (size_t)env;
    R[0] = cos(th); R[1] = -sin(th); R[2] = sin(th); R[3] = cos(th);
    if (s.done && clear_done) s.done[env] = 0;
}

__global__ void k_env_reset(f110_sim s, const double *__restrict__ poses, const uint8_t *__restrict__ mask) {
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= s.num_envs) return;
    if (mask && !mask[env]) return;
    env_counters_reset(s, env, poses + 3 * (size_t)env * s.num_agents);
}

// f110_env.py:294-302 + _check_done :204-246, one thread per env
__device__ __forceinline__ void env_post_step_one(const f110_sim &s, int env) {
    const int A = s.num_agents, NA = s.num_envs * s.num_agents;
    const double left_t = 2, right_t = 2;
    const double now = s.current_time[env] + s.timestep;
    s.current_time[env] = now;
    const double *R = s.start_rot + 4 * (size_t)env;
    bool all_done = true;
    for (int i = 0; i < A; i++) {
        const size_t a = (size_t)env * A + i;
        double px = s.state[a] - s.start_xs[a];
        double py = s.state[(size_t)NA + a] - s.start_ys[a];
        double dx = R[0] * px + R[1] * py;
        double ty = R[2] * px + R[3] * py;
        if (ty > left_t) ty -= left_t;
        else if (ty < -right_t) ty = -right_t - ty;
        else ty = 0;
        double dist2 = dx * dx + ty * ty;
        bool close = dist2 <= 0.1;
        int near = s.near_starts[a];
        double tog = s.toggle_list[a];
        if (close && !near) { near = 1; tog += 1; }
        else if (!close && near) { near = 0; tog += 1; }
        s.near_starts[a] = near;
        s.toggle_list[a] = tog;
        s.lap_counts[a] = floor(tog / 2);
        if (tog < 4) s.lap_times[a] = now;
        bool cp = tog >= 4;
        if (s.checkpoint_done) s.checkpoint_done[a] = cp ? 1 : 0;
        all_done = all_done && cp;
    }
    s.done[env] = ((s.collisions[(size_t)env * A + s.ego_idx] != 0.0) || all_done) ? 1 : 0;
}

__global__ void k_env_post_step(f110_sim s) {
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env < s.num_envs) env_post_step_one(s, env);
}

__device__ __forceinline__ uint64_t mix64(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

struct AutoResetArgs {
    const double *start_poses;   // [num_start][3] or NULL = off
    int num_start, pose_gap;
    uint64_t seed, tick_host;
};

// one thread per env: reset the env if its ego collided (benchmark / RL convenience, SURVEY.md 8d)
__device__ __forceinline__ void autoreset_one(const f110_sim &s, int env, const AutoResetArgs &ar) {
    const int A = s.num_agents, NA = s.num_envs * s.num_agents;
    if (s.collisions[(size_t)env * A + s.ego_idx] == 0.0) return;
    const double *__restrict__ start_poses = ar.start_poses;
    const int num_start = ar.num_start, pose_gap = ar.pose_gap;
    const uint64_t seed = ar.seed;
    const uint64_t tick = s.tick_counter ? (uint64_t)*s.tick_counter : ar.tick_host;
    uint64_t h = mix64(seed + 0x9E3779B97F4A7C15ull * (tick + 1) + 0xD1B54A32D192ED03ull * (uint64_t)(env + 1));
    int k = (int)((double)(h >> 11) * (1.0 / 9007199254740992.0) * num_start);
    if (k >= num_start) k = num_start - 1;
    double pose3[3 * 32];
    for (int i = 0; i < A; i++) {
        int kk = ((k - pose_gap * i) % num_start + num_start) % num_start;
        const size_t a = (size_t)env * A + i;
        const double x = start_poses[3 * kk], y = start_poses[3 * kk + 1], th = start_poses[3 * kk + 2];
        if (i < 32) { pose3[3 * i] = x; pose3[3 * i + 1] = y; pose3[3 * i + 2] = th; }
#pragma unroll
        for (int q = 0; q < 7; q++) s.state[(size_t)q * NA + a] = 0.0;
        s.state[a] = x;
        s.state[(size_t)NA + a] = y;
        s.state[(size_t)4 * NA + a] = th;
        s.steer_cnt[a] = 0;
        s.steer_buf[a] = 0.0;
        s.steer_buf[(size_t)NA + a] = 0.0;
        s.wall_flag[a] = 0;
        mark_march_cost_unknown(s, a);
    }
    if (s.current_time && A <= 32) env_counters_reset(s, env, pose3, false);
}

__global__ void k_autoreset(f110_sim s, AutoResetArgs ar) {
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env < s.num_envs) autoreset_one(s, env, ar);
}

// f110_tick: warp per agent; the warp that finishes an env last (per-env arrival counter) also runs the F110Env
// lap logic and the auto-reset for that env: k_finalize + k_env_post_step + k_autoreset in one launch
// MAXT / MINB: blocks of up to 4 agent-warps (A <= 4) are compiled without the 64-register cap of a 1024-thread block
template <int MAXT, int MINB>
__global__ void __launch_bounds__(MAXT, MINB) k_tail(f110_sim s, BeamView bv, int env_level, AutoResetArgs ar,
                                                      double max_scan_range, int envs_per_block) {
    // a block owns whole envs (blockDim = 32 * A * envs_per_block, A <= 32): the env-level step only needs what the
    // warps of its own block wrote, so a block barrier orders it -- no device-scope fence, no arrival atomics.  (The
    // first version had every warp execute __threadfence() + atomicAdd on a per-env counter; the fence's L1
    // invalidation (CCTL.IVALL) kept evicting the beam tables and poses of the other warps on the SM: 19 % of the
    // kernel's stall samples sat on the fences and 8 % on the scan-angle loads behind them.)
    const int A = s.num_agents;
    const int lane = threadIdx.x & 31;
    pdl_wait();                              // the march kernel (scans, wall flags) must be complete
    const int env0 = blockIdx.x * envs_per_block;
    const int a = env0 * A + (int)(threadIdx.x >> 5);
    if (a < s.num_envs * A) finalize_agent(s, bv, a, lane, max_scan_range);
    __syncthreads();
    if ((int)threadIdx.x < envs_per_block) {
        const int env = env0 + (int)threadIdx.x;
        if (env < s.num_envs) {
            if (env_level) env_post_step_one(s, env);
            if (ar.start_poses) autoreset_one(s, env, ar);
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) end_of_tick_housekeeping(s);
}

// ------------------------------------------------------------------------------------ k_tail2 (2 <= A <= 4)
// Same results as k_tail, reorganised (round 2).  ncu on k_tail at 16384 x 2: 1317 warp-instructions per agent, most of them the
// per-agent SCALAR prologue (opponent vertices, six atan2, asin, sqrt, nearest-beam searches) that all 32 lanes of the agent's
// warp execute redundantly (profiles/r2/finalize_cfg3_line_hot.txt).  Here a block owns EPB whole envs and works in three phases:
//   1. one THREAD per (ego, opponent) pair does the scalar prologue -- 32 pairs per warp instead of one -- and leaves a task
//      record in shared memory; one thread per agent also does the wall-hit zeroing, GJK and the collisions observation;
//   2. one WARP per ego walks its tasks and ray-casts the windows beam-parallel (the same loop as finalize_agent);
//   3. one thread per env: lap logic + auto-reset (as in k_tail).
struct TailTask {
    double px, py, yaw, phi, cone;
    double v[8];
    int lo, hi, active, pad;
};
#define F110_TAIL2_THREADS 256

__global__ void __launch_bounds__(F110_TAIL2_THREADS, 3) k_tail2(f110_sim s, BeamView bv, int env_level, AutoResetArgs ar,
                                                                  double max_scan_range, int envs_per_block) {
    extern __shared__ __align__(16) unsigned char tail2_smem[];
    TailTask *tasks = reinterpret_cast<TailTask *>(tail2_smem);
    const int A = s.num_agents, NA = s.num_envs * A;
    const int opp = A - 1;                                    // tasks per agent
    const int env0 = blockIdx.x * envs_per_block;
    const int envs_here = min(envs_per_block, s.num_envs - env0);
    const int agents_here = envs_here * A;
    const int ntasks = agents_here * opp;
    pdl_wait();                                                // the march kernel (scans, wall flags) must be complete

    // ---- phase 1: thread per (ego, opponent) pair
    for (int t = threadIdx.x; t < ntasks; t += blockDim.x) {
        const int la = t / opp, oj = t - la * opp;
        const int envl = la / A, slot = la - envl * A;
        const int env = env0 + envl, a = env * A + slot;
        const int j = oj < slot ? oj : oj + 1;                 // opponents in ascending index, skipping the ego itself
        const int hit = s.wall_flag[a];
        const double *pa = s.agent_poses + 5 * (size_t)a;
        const double px = pa[0], py = pa[1];
        // check_ttc zeroes state[3:] -- including the yaw -- before the opponent ray-cast reads it (:246-249, :225)
        const double yaw = hit ? 0.0 : pa[2];
        const double cyaw = hit ? 1.0 : pa[3], syaw = hit ? 0.0 : pa[4];
        const double *pb = s.agent_poses + 5 * (size_t)(env * A + j);
        if (oj == 0) {
            // per-agent duties: wall-hit zeroing, GJK against the other agents (collision_multiple :184-212), collisions obs
            if (hit) {
#pragma unroll
                for (int q = 0; q < 4; q++) s.state[(size_t)(3 + q) * NA + a] = 0.0;
            }
            int col = 0, cidx = -1;
            const double reach2 = (s.sim_length * s.sim_length + s.sim_width * s.sim_width) * 1.001;
            for (int jj = 0; jj < A; jj++) {
                if (jj == slot) continue;
                const double *pc = s.agent_poses + 5 * (size_t)(env * A + jj);
                const double ddx = pc[0] - pa[0], ddy = pc[1] - pa[1];
                if (ddx * ddx + ddy * ddy > reach2) continue;
                double vme[8], vo[8];
                get_vertices_cs(pa[0], pa[1], pa[3], pa[4], s.sim_length, s.sim_width, vme);
                get_vertices_cs(pc[0], pc[1], pc[3], pc[4], s.sim_length, s.sim_width, vo);
                const bool c = (slot < jj) ? gjk_collision(vme, vo) : gjk_collision(vo, vme);
                if (c) { col = 1; cidx = max(cidx, jj); }
            }
            s.collisions[a] = (col || hit) ? 1.0 : 0.0;
            s.collision_idx[a] = cidx;
        }
        // ray_cast_agents (:206-227): the scalar part of one opponent
        TailTask &k = tasks[t];
        const double *p = s.params + (size_t)(s.params_per_env ? a : slot) * F110_NPARAM;
        const double length = p[P_LENGTH], width = p[P_WIDTH];
        const double half_diag = 0.5 * sqrt(length * length + width * width);
        const double ddx = pb[0] - px, ddy = pb[1] - py;
        const double far = max_scan_range + half_diag;
        int active = 1;
        if (ddx * ddx + ddy * ddy > far * far) active = 0;     // cannot shorten any beam (see finalize_agent)
        k.active = active;
        if (active) {
            double v[8];
            get_vertices_cs(pb[0], pb[1], pb[3], pb[4], length, width, v);
            int lo, hi;
            double phi;
            blocked_view_indices_cs(px, py, cyaw, syaw, v, bv.scan_angles, bv.num_beams, bv.fov, bv.angle_increment, pb[0], pb[1],
                                    lo, hi, phi);
            double cone = 4.0;
            if (hi - lo >= 96) {
                const double dist = sqrt(ddx * ddx + ddy * ddy);
                if (dist > 1.25 * half_diag) cone = asin(half_diag / dist) + 0.05;
            }
            k.px = px; k.py = py; k.yaw = yaw; k.phi = phi; k.cone = cone; k.lo = lo; k.hi = hi;
#pragma unroll
            for (int q = 0; q < 8; q++) k.v[q] = v[q];
        }
    }
    __syncthreads();

    // ---- phase 2: warp per ego, its opponents one after the other (they update the same scan)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    for (int la = warp; la < agents_here; la += nwarps) {
        const int a = env0 * A + la;
        float *scan = s.scans + (size_t)a * bv.num_beams;
        for (int oj = 0; oj < opp; oj++) {
            const TailTask &k = tasks[la * opp + oj];
            if (!k.active) continue;
            const double px = k.px, py = k.py, yaw = k.yaw, phi = k.phi, cone = k.cone;
            const int lo = k.lo, hi = k.hi;
            double v[8];
#pragma unroll
            for (int q = 0; q < 8; q++) v[q] = k.v[q];
            auto cast_beams = [&](int i0, int i1) {
                for (int i = i0 + lane; i <= i1; i += 32) {
                    const float cur = scan[i];
                    double bt = yaw + bv.scan_angles[i];
                    double dl = bt - phi;
                    dl = dl - (2 * M_PI) * rint(dl * (1.0 / (2 * M_PI)));
                    const double adl = fabs(dl);
                    if (adl > cone && (M_PI - adl) > cone) continue;
                    double v3x, v3y;
                    sincos(bt + M_PI / 2., &v3y, &v3x);
                    const double curd = (double)cur;
                    double r = INFINITY;
#pragma unroll
                    for (int e = 0; e < 4; e++) {
                        int e2 = (e + 1) & 3;
                        double d = get_range_below(px, py, v3x, v3y, v[2 * e], v[2 * e + 1], v[2 * e2], v[2 * e2 + 1], curd);
                        if (d < r) r = d;
                    }
                    float rf = (float)r;
                    if (rf < cur) scan[i] = rf;
                }
            };
            if (cone < 3.5 && hi - lo >= 96) {
                const double base = phi - yaw, half = bv.fov / 2., inv_inc = 1.0 / bv.angle_increment;
                const int m0 = max(-3, (int)floor((-half - cone - 0.02 - base) * (1.0 / M_PI))),
                          m1 = min(5, (int)ceil((half + cone + 0.02 - base) * (1.0 / M_PI)));
                for (int m = m0; m <= m1; m++) {
                    const double c = base + (double)m * M_PI;
                    const double f0 = (c - cone + half) * inv_inc - 2.0, f1 = (c + cone + half) * inv_inc + 2.0;
                    if (f1 < (double)lo || f0 > (double)hi) continue;
                    const int i0 = max(lo, (int)floor(fmax(f0, (double)lo))), i1 = min(hi, (int)ceil(fmin(f1, (double)hi)));
                    cast_beams(i0, i1);
                }
            } else {
                cast_beams(lo, hi);
            }
            __syncwarp();
        }
    }
    __syncthreads();

    // ---- phase 3: env level
    if ((int)threadIdx.x < envs_here) {
        const int env = env0 + (int)threadIdx.x;
        if (env_level) env_post_step_one(s, env);
        if (ar.start_poses) autoreset_one(s, env, ar);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) end_of_tick_housekeeping(s);
}

// ------------------------------------------------------------------------------------ standalone kernels
__global__ void k_rhs(const double *__restrict__ x, const double *__restrict__ u, const double *__restrict__ p,
                      int M, double *__restrict__ f) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    double xs[7], fs[7];
    for (int k = 0; k < 7; k++) xs[k] = x[7 * (size_t)i + k];
    vehicle_dynamics_st(xs, u[2 * (size_t)i], u[2 * (size_t)i + 1], p, fs);
    for (int k = 0; k < 7; k++) f[7 * (size_t)i + k] = fs[k];
}

__global__ void k_rhs_ks(const double *__restrict__ x, const double *__restrict__ u, const double *__restrict__ p,
                         int M, double *__restrict__ f) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    double xs[5], fs[5];
    for (int k = 0; k < 5; k++) xs[k] = x[5 * (size_t)i + k];
    vehicle_dynamics_ks(xs, u[2 * (size_t)i], u[2 * (size_t)i + 1], p, fs);
    for (int k = 0; k < 5; k++) f[5 * (size_t)i + k] = fs[k];
}

__global__ void k_pid(const double *__restrict__ in, const double *__restrict__ p, int M, double *__restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    double accl, sv;
    pid(in[4 * (size_t)i], in[4 * (size_t)i + 1], in[4 * (size_t)i + 2], in[4 * (size_t)i + 3], p[P_SVMAX],
        p[P_AMAX], p[P_VMAX], p[P_VMIN], accl, sv);
    out[2 * (size_t)i] = accl;
    out[2 * (size_t)i + 1] = sv;
}

__global__ void k_vertices(const double *__restrict__ poses, double length, double width, int M,
                           double *__restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    double v[8];
    get_vertices(poses[3 * (size_t)i], poses[3 * (size_t)i + 1], poses[3 * (size_t)i + 2], length, width, v);
    for (int k = 0; k < 8; k++) out[8 * (size_t)i + k] = v[k];
}

__global__ void k_gjk(const double *__restrict__ va, const double *__restrict__ vb, int M, int32_t *__restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    double a[8], b[8];
    for (int k = 0; k < 8; k++) { a[k] = va[8 * (size_t)i + k]; b[k] = vb[8 * (size_t)i + k]; }
    out[i] = gjk_collision(a, b) ? 1 : 0;
}

__global__ void k_gjk_multiple(const double *__restrict__ verts, int M, int n, double *__restrict__ collisions,
                               double *__restrict__ collision_idx) {
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= M) return;
    const double *V = verts + (size_t)e * n * 8;
    for (int i = 0; i < n; i++) { collisions[(size_t)e * n + i] = 0.; collision_idx[(size_t)e * n + i] = -1.; }
    for (int i = 0; i < n - 1; i++)
        for (int j = i + 1; j < n; j++) {
            double a[8], b[8];
            for (int k = 0; k < 8; k++) { a[k] = V[8 * i + k]; b[k] = V[8 * j + k]; }
            if (gjk_collision(a, b)) {
                collisions[(size_t)e * n + i] = 1.; collisions[(size_t)e * n + j] = 1.;
                collision_idx[(size_t)e * n + i] = j; collision_idx[(size_t)e * n + j] = i;
            }
        }
}

__global__ void k_check_ttc(BeamView bv, const double *__restrict__ scans, const double *__restrict__ vel,
                            double thresh, int M, int32_t *__restrict__ out) {
    const int a = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (a >= M) return;
    int hit = 0;
    for (int i = lane; i < bv.num_beams; i += 32)
        hit |= ttc_hit(scans[(size_t)a * bv.num_beams + i], vel[a], bv.cosines[i], bv.side_distances[i], thresh) ? 1 : 0;
    hit = __any_sync(0xffffffffu, hit);
    if (lane == 0) out[a] = hit ? 1 : 0;
}

__global__ void k_ray_cast(BeamView bv, const double *__restrict__ poses, const double *__restrict__ opp, int M,
                           float *__restrict__ scans, int32_t *__restrict__ window) {
    const int a = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (a >= M) return;
    const double px = poses[3 * (size_t)a], py = poses[3 * (size_t)a + 1], yaw = poses[3 * (size_t)a + 2];
    double v[8];
    for (int k = 0; k < 8; k++) v[k] = opp[8 * (size_t)a + k];
    int lo, hi;
    blocked_view_indices(px, py, yaw, v, bv.scan_angles, bv.num_beams, bv.fov, bv.angle_increment, lo, hi);
    if (window && lane == 0) { window[2 * a] = lo; window[2 * a + 1] = hi; }
    float *scan = scans + (size_t)a * bv.num_beams;
    for (int i = lo + lane; i <= hi; i += 32) {
        double bt = yaw + bv.scan_angles[i];
        double v3x = cos(bt + M_PI / 2.), v3y = sin(bt + M_PI / 2.);
        double r = INFINITY;
        for (int e = 0; e < 4; e++) {
            int e2 = (e + 1) & 3;
            double d = get_range(px, py, v3x, v3y, v[2 * e], v[2 * e + 1], v[2 * e2], v[2 * e2 + 1]);
            if (d < r) r = d;
        }
        float rf = (float)r;
        if (rf < scan[i]) scan[i] = rf;
    }
}

// four ranges -> three 32-bit words (12 bytes): 24-bit fixed point with 2^-19 m steps
__global__ void k_pack_u24(const float *__restrict__ scans, long long count, uint8_t *__restrict__ out) {
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long i0 = g * 4;
    if (i0 >= count) return;
    unsigned q[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const float r = (i0 + k < count) ? scans[i0 + k] : 0.0f;
        const float v = fminf(fmaxf(r, 0.0f) * 524288.0f, 16777215.0f);      // 2^19; exact scaling, then round to nearest
        q[k] = (unsigned)__float2uint_rn(v);
    }
    if (i0 + 4 <= count && ((i0 * 3) & 3) == 0) {
        unsigned *o = reinterpret_cast<unsigned *>(out + i0 * 3);
        o[0] = q[0] | (q[1] << 24);
        o[1] = (q[1] >> 8) | (q[2] << 16);
        o[2] = (q[2] >> 16) | (q[3] << 8);
    } else {
        for (int k = 0; k < 4 && i0 + k < count; k++) {
            uint8_t *o = out + (i0 + k) * 3;
            o[0] = (uint8_t)q[k]; o[1] = (uint8_t)(q[k] >> 8); o[2] = (uint8_t)(q[k] >> 16);
        }
    }
}

__global__ void k_scan_noise(float *__restrict__ scans, long long count, double std_dev, uint64_t seed,
                             uint64_t offset) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    scans[i] = (float)((double)scans[i] + std_dev * normal_sample(seed, 0xFFFFFFFFull, offset + (uint64_t)i));
}

static int check_sim(const f110_sim *s) {
    if (!s) return F110_ERR_INVALID;
    if (s->num_envs <= 0 || s->num_agents <= 0) return F110_ERR_INVALID;
    if (s->integrator != 1 && s->integrator != 2) return F110_ERR_INTEGRATOR;
    if (!s->params || !s->state || !s->steer_buf || !s->steer_cnt || !s->scan_pose || !s->agent_poses ||
        !s->scans || !s->wall_flag || !s->collisions || !s->collision_idx)
        return F110_ERR_INVALID;
    return F110_OK;
}
static int check_map(const f110_map *m) {
    if (!m) return F110_ERR_INVALID;
    if (!m->dt || m->height <= 0 || m->width <= 0) return F110_ERR_NO_MAP;
    if (!m->sines || !m->cosines || m->theta_dis <= 0 || !(m->resolution > 0)) return F110_ERR_INVALID;
    return F110_OK;
}
static int check_beams(const f110_beams *b) {
    if (!b || b->num_beams <= 1 || !b->scan_angles || !b->cosines || !b->side_distances) return F110_ERR_INVALID;
    return F110_OK;
}

static unsigned long long *g_trace = nullptr;
static unsigned long long *g_tile_counter = nullptr;   // debug only: lookups served from the shared-memory tile   // debug only: per-block timeline buffer (f110_debug_set_trace)

static int num_sms() {
    static int n = 0;
    if (n <= 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
            n = 148;
    }
    return n;
}

// A/B switch for measurements (profiles/r2/README.md; f110_debug_set_variant or F110_MARCH_VARIANT): 0 = default (k_march_lean,
// fp64 table, half of the queue dynamic); 66 / 60 / 61 = static dealing with 4 x 512 / 2 x 1024 / 8 x 256 threads per SM;
// 40 / 41 / 42 = dynamic with 4 x 512 / 3 x 512 / 2 x 1024; 20 / 22 = rank-coded table + shared LUT; 21 = 48 warps/SM;
// 30 / 31 = TMA tile 128 / 160 cells; 62-65 = thread-block clusters sharing a ticket counter; 1 / 6 = round-1 persistent kernel
// (fp64 / coded); 7 / 9 = no queue (block per 64-beam tile); 13 = the literal k_raymarch
static int g_variant = -1, g_chunk = -1;
// Dynamic second half of the queue (k_march_lean<DYN>): every block gets g_dyn_pct % of its fair share dealt statically and claims
// the rest in runs from one global counter, g_dyn_ahead runs ahead of their use.  50 % / 4 is the measured optimum (cfg3 march
// 419 -> 407 us, cfg2x2 116 -> 113.6, cfg2 68.5 -> 68.1; profiles/r2/ab_march_11..13_*.jsonl): the default of variant 0.
static int g_dyn_pct = 50, g_dyn_ahead = 4;
static int g_ipt[4] = {-1, -1, -1, 255};  // log2(entries per ticket): very heavy, heavy, light runs, dynamic tail (255 = by the class it starts in); -1 = by queue length
static int rm_variant() {
    if (g_variant < 0) {
        const char *e = getenv("F110_MARCH_VARIANT");
        g_variant = e ? atoi(e) : 0;
    }
    return g_variant;
}

static int launch_raymarch(const MapView &mv, const BeamView &bv, const MarchArgs &g, bool fast, bool standalone,
                           cudaStream_t st) {
    const int threads = 256;
    const long long blocks = (g.total + threads - 1) / threads;
    if (blocks <= 0 || blocks > 0x7fffffffll) return F110_ERR_INVALID;
    if (fast) {
        if (standalone) k_raymarch<true, true><<<(unsigned)blocks, threads, 0, st>>>(mv, bv, g);
        else k_raymarch<true, false><<<(unsigned)blocks, threads, 0, st>>>(mv, bv, g);
    } else {
        if (standalone) k_raymarch<false, true><<<(unsigned)blocks, threads, 0, st>>>(mv, bv, g);
        else k_raymarch<false, false><<<(unsigned)blocks, threads, 0, st>>>(mv, bv, g);
    }
    LAUNCH_CHECK("k_raymarch");
    return F110_OK;
}

template <int PT, int SUB, bool CELLS>
static void launch_persistent(const MarchK &k, const MarchQueue &mq, unsigned blocks, bool coded, bool noise, bool count,
                              cudaStream_t st) {
    if (k.trace) {
        if (coded && CELLS) k_march_persistent<CELLS, false, false, true, PT, SUB, CELLS><<<blocks, PT, 0, st>>>(k, mq);
        else k_march_persistent<false, false, false, true, PT, SUB, CELLS><<<blocks, PT, 0, st>>>(k, mq);
    } else if (coded && CELLS) {
        if (count) k_march_persistent<CELLS, false, true, false, PT, SUB, CELLS><<<blocks, PT, 0, st>>>(k, mq);
        else if (noise) k_march_persistent<CELLS, true, false, false, PT, SUB, CELLS><<<blocks, PT, 0, st>>>(k, mq);
        else k_march_persistent<CELLS, false, false, false, PT, SUB, CELLS><<<blocks, PT, 0, st>>>(k, mq);
    } else {
        if (count) k_march_persistent<false, false, true, false, PT, SUB, CELLS><<<blocks, PT, 0, st>>>(k, mq);
        else if (noise) k_march_persistent<false, true, false, false, PT, SUB, CELLS><<<blocks, PT, 0, st>>>(k, mq);
        else k_march_persistent<false, false, false, false, PT, SUB, CELLS><<<blocks, PT, 0, st>>>(k, mq);
    }
}

// Launch with the programmatic-stream-serialization attribute (PDL) when enabled: the kernel may become resident before
// its predecessor in the stream has finished and synchronises itself with pdl_wait().
// measured (profiles/r2/ab_march_5_pdl_tail.jsonl): inside a CUDA graph PDL wins nothing (cfg2 85.9 vs 86.0-88.0 us, cfg3 563-573 vs
// 560-569 us), so it is off by default and kept as a switch (f110_debug_set_pdl); k_tail is fastest with the 64-register
// budget (occupancy beats spills: cfg3 560.0 / 565.1 / 569.3 us for 64 / 96 / 128 registers)
static int g_pdl = 0;
static int g_tail_minb = 8;
static int g_tail2_threads = F110_TAIL2_THREADS, g_tail2_agents = 64;    // block shape of k_tail2 (f110_debug_set_tail2)
static int g_tail2_forced = 0;                                            // agents per block forced exactly (debug setter, agents > 64 or < 0)
static int g_tail2 = 1;          // 2 <= A <= 4: the two-phase k_tail2 (f110_debug_set_tail(-1) switches back to k_tail for the A/B)
static thread_local bool g_pdl_this_step = false;     // set by step_impl: PDL only when no events are recorded between the kernels
template <typename... KArgs, typename... Args>
static void launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = (pdl && g_pdl) ? 1 : 0;
    cudaLaunchKernelEx(&cfg, kernel, args...);
}
// launch in thread-block clusters of `cl` CTAs (grid must be a multiple of cl)
template <typename... KArgs, typename... Args>
static void launch_cluster(void (*kernel)(KArgs...), dim3 grid, dim3 block, unsigned cl, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = 0; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = cl; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, kernel, args...);
}
// does a grid of `blocks` CTAs in clusters of CL fit on the device at once?  (a persistent kernel needs all of them resident)
template <typename K>
static bool clusters_fit(K kernel, unsigned blocks, unsigned threads, unsigned cl) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(blocks); cfg.blockDim = dim3(threads); cfg.dynamicSmemBytes = 0;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = cl; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, kernel, &cfg) != cudaSuccess) { cudaGetLastError(); return false; }
    return (unsigned)n * cl >= blocks;
}

template <int TABLE, bool CELLS, bool LAYERED, int MINB, bool DYN = false, int PT = 512, int IPT = 1, int RING = 0>
static void launch_lean_t(const LeanK &q, const MarchQueue &mq, unsigned blocks, bool noise, bool count, cudaStream_t st) {
    const bool pdl = g_pdl_this_step;
    if (count) launch_k(k_march_lean<TABLE, false, true, CELLS, LAYERED, PT, MINB, DYN, 1, IPT, RING>, dim3(blocks), dim3(PT), 0, st, pdl, q, mq);
    else if (noise) launch_k(k_march_lean<TABLE, true, false, CELLS, LAYERED, PT, MINB, DYN, 1, IPT, RING>, dim3(blocks), dim3(PT), 0, st, pdl, q, mq);
    else launch_k(k_march_lean<TABLE, false, false, CELLS, LAYERED, PT, MINB, DYN, 1, IPT, RING>, dim3(blocks), dim3(PT), 0, st, pdl, q, mq);
}
static void launch_lean(const LeanK &q, const MarchQueue &mq, unsigned sms, bool cells, bool coded, bool occ3, bool layered,
                        bool noise, bool count, bool dyn, cudaStream_t st) {
    // thread-block clusters sharing one ticket counter (variants 62-65), plain noise-free marching only
    if (cells && !layered && !coded && !noise && !count && rm_variant() >= 62 && rm_variant() <= 65) {
        const int v = rm_variant();
        bool ok = false;
        if (v == 62) { auto k = k_march_lean<0, false, false, true, false, 1024, 2, false, 4>;
                       if ((ok = clusters_fit(k, sms * 2u / 4u * 4u, 1024, 4))) launch_cluster(k, dim3(sms * 2u / 4u * 4u), dim3(1024), 4, st, q, mq); }
        if (v == 63) { auto k = k_march_lean<0, false, false, true, false, 1024, 2, false, 2>;
                       if ((ok = clusters_fit(k, sms * 2u, 1024, 2))) launch_cluster(k, dim3(sms * 2u), dim3(1024), 2, st, q, mq); }
        if (v == 64) { auto k = k_march_lean<0, false, false, true, false, 512, 4, false, 4>;
                       if ((ok = clusters_fit(k, sms * 4u, 512, 4))) launch_cluster(k, dim3(sms * 4u), dim3(512), 4, st, q, mq); }
        if (v == 65) { auto k = k_march_lean<0, false, false, true, false, 512, 4, false, 8>;
                       if ((ok = clusters_fit(k, sms * 4u / 8u * 8u, 512, 8))) launch_cluster(k, dim3(sms * 4u / 8u * 8u), dim3(512), 8, st, q, mq); }
        if (ok) return;
        if (getenv("F110_DEBUG")) fprintf(stderr, "f110: cluster variant %d does not fit, using the default launch\n", v);
    }
    // Block shape at the same 64 warps/SM.  Two 1024-thread blocks per SM (32 warps share a ticket counter, the queue is dealt
    // to half as many blocks) beat four 512-thread blocks whenever a block gets enough items -- cfg3 march 443 -> 420 us,
    // cfg5_2160 819 -> 761, cfg2x2 120.2 -> 116.2 -- and lose when it does not: cfg2 (470 items per big block) 68.2 -> 70.5 us
    // (profiles/r2/ab_march_7_*.jsonl, ab_march_8_*.jsonl).  Variant 60 / 61 / 66 force 2 x 1024 / 8 x 256 / 4 x 512.
    const int v = rm_variant();
    const bool big = (v == 60) || (v != 61 && v != 66 && v != 44 && v != 21 && v != 22 && !dyn && !coded && !occ3 &&
                                   (unsigned long long)mq.items >= 700ull * 2ull * (unsigned long long)sms);
    if (big && !coded) {
        if (!cells && layered) launch_lean_t<0, false, true, 2, false, 1024>(q, mq, sms * 2u, noise, count, st);
        else if (!cells) launch_lean_t<0, false, false, 2, false, 1024>(q, mq, sms * 2u, noise, count, st);
        else if (layered) launch_lean_t<0, true, true, 2, false, 1024>(q, mq, sms * 2u, noise, count, st);
        else launch_lean_t<0, true, false, 2, false, 1024>(q, mq, sms * 2u, noise, count, st);
        return;
    }
    if (cells && !layered && !coded && v == 61) { launch_lean_t<0, true, false, 8, false, 256>(q, mq, sms * 8u, noise, count, st); return; }
    // two queue entries per ticket (variant 43: dynamic, 4 x 512; 44: static, 4 x 512); needs runs of >= 2 entries
    if (cells && !layered && !coded && mq.chunk_shift >= 1 && v == 43 && dyn) { launch_lean_t<0, true, false, 4, true, 512, 2>(q, mq, sms * 4u, noise, count, st); return; }
    if (cells && !layered && !coded && mq.chunk_shift >= 2 && v == 45 && dyn) { launch_lean_t<0, true, false, 4, true, 512, 4>(q, mq, sms * 4u, noise, count, st); return; }
    if (cells && !layered && !coded && mq.chunk_shift >= 1 && v == 44) { launch_lean_t<0, true, false, 4, false, 512, 2>(q, mq, sms * 4u, noise, count, st); return; }
    // ring hand-off through shared atomics (81 / 83 / 85: 4 / 2 entries per ticket / by run class) and through st.release / ld.acquire
    // (82 / 84 / 86)
    if (dyn && cells && !layered && !coded && mq.chunk_shift >= 3) {
        if (v == 81) { launch_lean_t<0, true, false, 4, true, 512, 4, 1>(q, mq, sms * 4u, noise, count, st); return; }
        if (v == 82) { launch_lean_t<0, true, false, 4, true, 512, 4, 2>(q, mq, sms * 4u, noise, count, st); return; }
        if (v == 83) { launch_lean_t<0, true, false, 4, true, 512, 2, 1>(q, mq, sms * 4u, noise, count, st); return; }
        if (v == 84) { launch_lean_t<0, true, false, 4, true, 512, 2, 2>(q, mq, sms * 4u, noise, count, st); return; }
        if (v == 85) { launch_lean_t<0, true, false, 4, true, 512, 0, 1>(q, mq, sms * 4u, noise, count, st); return; }
        if (v == 86) { launch_lean_t<0, true, false, 4, true, 512, 0, 2>(q, mq, sms * 4u, noise, count, st); return; }
    }
    // 48 warps per SM (3 x 512 threads, 40 registers) with 4 / 2 entries per ticket
    if (dyn && cells && !layered && !coded && mq.chunk_shift >= 3 && v == 57) { launch_lean_t<0, true, false, 3, true, 512, 4>(q, mq, sms * 3u, noise, count, st); return; }
    if (dyn && cells && !layered && !coded && mq.chunk_shift >= 2 && v == 58) { launch_lean_t<0, true, false, 3, true, 512, 2>(q, mq, sms * 3u, noise, count, st); return; }
    if (dyn && cells && !layered && !coded && v == 42) { launch_lean_t<0, true, false, 2, true, 1024>(q, mq, sms * 2u, noise, count, st); return; }
    if (dyn && cells && !layered && !coded) {
        if (occ3) launch_lean_t<0, true, false, 3, true>(q, mq, sms * 3u, noise, count, st);
        else if (v == 40) launch_lean_t<0, true, false, 4, true>(q, mq, sms * 4u, noise, count, st);       // one entry per ticket, compile-time
        // Long queues (>= 72 entries per warp: cfg3, the beam sweep): four entries per ticket throughout, fixed at compile time --
        // cfg3 march 368 us against 378 with the very heavy runs dealt one or two entries at a time, 407 with one entry per
        // ticket everywhere.  Shorter queues: ticket size by the class of the run (dyn_queue_position_zoned), which is what
        // keeps four very heavy entries from landing on one warp (uniform 4: cfg2x2 139 us instead of 112, cfg2 122 instead of 68).
        // Medium queues (27..72 entries per warp: cfg2x2, n12288a1): two entries per ticket (cfg2x2 109-110 us against 111 by class).
        // The ring words go through st.release / ld.acquire (RING = 2; the volatile formulation times the same, the one in
        // shared atomics that racecheck accepts costs 13 %: profiles/r2/ab_march_28_ring_handoff.jsonl).
        else if (mq.uniform_ipt4 == 4u && v == 0) launch_lean_t<0, true, false, 4, true, 512, 4, 2>(q, mq, sms * 4u, noise, count, st);
        else if (mq.uniform_ipt4 == 2u && v == 0) launch_lean_t<0, true, false, 4, true, 512, 2, 2>(q, mq, sms * 4u, noise, count, st);
        else launch_lean_t<0, true, false, 4, true, 512, 0, 2>(q, mq, sms * 4u, noise, count, st);
        return;
    }
    if (dyn && !cells && !layered) { launch_lean_t<0, false, false, 4, true, 512, 0, 2>(q, mq, sms * 4u, noise, count, st); return; }
    if (!cells && layered) launch_lean_t<0, false, true, 4>(q, mq, sms * 4u, noise, count, st);
    else if (!cells) launch_lean_t<0, false, false, 4>(q, mq, sms * 4u, noise, count, st);
    else if (layered) launch_lean_t<0, true, true, 4>(q, mq, sms * 4u, noise, count, st);
    else if (coded && occ3) launch_lean_t<1, true, false, 3>(q, mq, sms * 3u, noise, count, st);
    else if (coded) launch_lean_t<1, true, false, 4>(q, mq, sms * 4u, noise, count, st);
    else if (occ3) launch_lean_t<0, true, false, 3>(q, mq, sms * 3u, noise, count, st);
    else launch_lean_t<0, true, false, 4>(q, mq, sms * 4u, noise, count, st);
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link against libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

template <int TILE, int NSLOT>
static int launch_tile_t(const TileK &t, const f110_map *map, unsigned sms, bool noise, bool count, cudaStream_t st) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) return cuda_fail(cudaErrorNotSupported, "cuTensorMapEncodeTiled entry point");
    CUtensorMap tm;
    const cuuint64_t dims[2] = { (cuuint64_t)map->codes_pitch, (cuuint64_t)(map->height + 1) };
    const cuuint64_t strides[1] = { (cuuint64_t)map->codes_pitch };
    const cuuint32_t box[2] = { (cuuint32_t)TILE, (cuuint32_t)TILE };
    const cuuint32_t estr[2] = { 1u, 1u };
    const CUresult r = enc(&tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, (void *)map->dt_codes_pad, dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return cuda_fail(cudaErrorInvalidValue, "cuTensorMapEncodeTiled");
    const size_t smem = sizeof(TileSmem<TILE, NSLOT>);
    constexpr int PT = 512;
    constexpr int MINB = 4;
    if (count) {
        CUDA_TRY(cudaFuncSetAttribute(k_march_tile<false, true, TILE, NSLOT, PT, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_march_tile<false, true, TILE, NSLOT, PT, MINB><<<sms * MINB, PT, smem, st>>>(t, tm);
    } else if (noise) {
        CUDA_TRY(cudaFuncSetAttribute(k_march_tile<true, false, TILE, NSLOT, PT, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_march_tile<true, false, TILE, NSLOT, PT, MINB><<<sms * MINB, PT, smem, st>>>(t, tm);
    } else {
        CUDA_TRY(cudaFuncSetAttribute(k_march_tile<false, false, TILE, NSLOT, PT, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_march_tile<false, false, TILE, NSLOT, PT, MINB><<<sms * MINB, PT, smem, st>>>(t, tm);
    }
    return F110_OK;
}
static int launch_tile(const TileK &t, const f110_map *map, int tile_sz, unsigned sms, bool noise, bool count, cudaStream_t st) {
    if (tile_sz == 160) return launch_tile_t<160, 2>(t, map, sms, noise, count, st);
    return launch_tile_t<128, 3>(t, map, sms, noise, count, st);
}

template <int MINB, bool CELLS>
static void launch_march(const MarchK &k, dim3 grid, bool coded, bool noise, bool count, cudaStream_t st) {
    if (coded && CELLS) {
        if (count) k_march<CELLS, false, true, MINB, CELLS><<<grid, 64, 0, st>>>(k);
        else if (noise) k_march<CELLS, true, false, MINB, CELLS><<<grid, 64, 0, st>>>(k);
        else k_march<CELLS, false, false, MINB, CELLS><<<grid, 64, 0, st>>>(k);
    } else {
        if (count) k_march<false, false, true, MINB, CELLS><<<grid, 64, 0, st>>>(k);
        else if (noise) k_march<false, true, false, MINB, CELLS><<<grid, 64, 0, st>>>(k);
        else k_march<false, false, false, MINB, CELLS><<<grid, 64, 0, st>>>(k);
    }
}

}  // namespace f110

using namespace f110;

// ================================================================================== C ABI
extern "C" {

int f110_abi_version(void) { return F110_ABI_VERSION; }

/* debug aid (not in the public header): device buffer [blocks][4] u64 that the march kernels fill with
 * (smid, start ns, end ns, max steps of warp 0) per block; NULL switches it off. */
void f110_debug_set_trace(unsigned long long *buf) { g_trace = buf; }
/* measurement aid (not in the public header): select the march kernel variant at run time (tools/ab_march.py) */
void f110_debug_set_variant(int variant) { g_variant = variant < 0 ? 0 : variant; }
void f110_debug_set_dyn(int static_pct, int ahead) {
    g_dyn_pct = static_pct < 0 ? 0 : (static_pct > 100 ? 100 : static_pct);
    g_dyn_ahead = ahead < 1 ? 1 : (ahead > 8 ? 8 : ahead);
}
/* log2(queue entries per ticket) for runs of very heavy / heavy / light entries and for the dynamic tail of the default launch
 * (dyn_tail < 0: by the class the tail starts in) */
void f110_debug_set_ipt(int very_heavy, int heavy, int light, int dyn_tail) {
    const int v[4] = {very_heavy, heavy, light, dyn_tail};
    for (int z = 0; z < 4; z++) g_ipt[z] = (v[z] < 0 || v[z] > 3) ? (z == 3 ? 255 : -1) : v[z];
}
void f110_debug_set_pdl(int on) { g_pdl = on ? 1 : 0; }
void f110_debug_set_tail2(int threads, int agents) {
    g_tail2_threads = (threads >= 32 && threads <= F110_TAIL2_THREADS) ? (threads / 32) * 32 : F110_TAIL2_THREADS;
    g_tail2_forced = (agents > 64 || agents < 0) ? 1 : 0;
    if (agents < 0) agents = -agents;
    g_tail2_agents = (agents >= 4 && agents <= 128) ? agents : 64;
}
void f110_debug_set_tail(int minb) {      // -1: k_tail always; -2 or a register budget: k_tail2 for 2 <= A <= 4 (the default)
    if (minb == -1) { g_tail2 = 0; g_tail_minb = 8; }
    else if (minb == -2) { g_tail2 = 1; g_tail_minb = 8; }
    else { g_tail2 = 1; g_tail_minb = minb; }
}
void f110_debug_set_tile_counter(unsigned long long *buf) { g_tile_counter = buf; }
void f110_debug_set_chunk(int chunk_shift) { g_chunk = (chunk_shift < 0 || chunk_shift > 6) ? 3 : chunk_shift; }

const char *f110_status_string(int status) {
    switch (status) {
        case F110_OK: return "ok";
        case F110_ERR_INVALID: return "invalid argument";
        case F110_ERR_NO_MAP: return "Map is not set for scan simulator.";
        case F110_ERR_CUDA: return "CUDA runtime error";
        case F110_ERR_INTEGRATOR: return "Invalid Integrator Specified. Please choose RK4 or Euler";
        case F110_ERR_POSE_COUNT: return "Number of poses for reset does not match number of agents.";
        case F110_ERR_AGENT_INDEX: return "Index given is out of bounds for list of agents.";
        default: return "unknown status";
    }
}

const char *f110_last_cuda_error(void) { return g_cuda_err; }

struct TailOpts {
    bool fused;              // k_tail instead of k_finalize
    int env_level;
    AutoResetArgs ar;
};

static int step_impl(const f110_sim *sim, const f110_map *map, const f110_beams *beams, const double *actions,
                     cudaStream_t st, cudaEvent_t *ev /* NULL or [4] */, const TailOpts *tail = nullptr) {
    int rc;
    if ((rc = check_sim(sim)) || (rc = check_map(map)) || (rc = check_beams(beams))) return rc;
    if (!actions) return F110_ERR_INVALID;
    // argument combinations are rejected BEFORE anything is enqueued: a tick either runs completely or not at all
    if (sim->lookup_counter && sim->noise_std > 0.0) return F110_ERR_INVALID;   // counting runs are noise-free by construction
    if ((long long)sim->num_envs * sim->num_agents > 0x7fffffffll) return F110_ERR_INVALID;
    const int NA = sim->num_envs * sim->num_agents;
    const MapView mv = make_view(map);
    const BeamView bv = make_view(beams);

    if (ev) CUDA_TRY(cudaEventRecord(ev[0], st));
    g_pdl_this_step = (ev == nullptr);
    const int variant = rm_variant();
    // work-item width: march_ipa = ceil(B/32) -> one 32-beam slice per item, ceil(B/64) -> two
    const int item_sub = (sim->march_ipa == (beams->num_beams + 31) / 32) ? 1
                       : (sim->march_ipa == (beams->num_beams + 63) / 64) ? 2 : 0;
    const bool queued = sim->march_cost && sim->march_order && sim->march_count && variant != 7 &&
                        item_sub != 0 && sim->march_ipa <= 256 &&
                        (unsigned long long)NA < (1ull << 22) &&
                        map->orig_c == 1.0 && map->orig_s == 0.0 && map->sincos && beams->cos_side && variant != 13;
    const int dyn_blocks = (NA + 127) / 128;
    int order_blocks = queued ? (int)(((long long)NA * sim->march_ipa + 128 * F110_ORDER_ITEMS_PER_THREAD - 1) /
                                         (128 * F110_ORDER_ITEMS_PER_THREAD)) : 0;
    // the lean march kernels need an unrotated map origin and the interleaved tables; cell units additionally a
    // power-of-two resolution (fast_path) and the cell-unit table
    const bool cell_march = map->orig_c == 1.0 && map->orig_s == 0.0 && map->sincos && beams->cos_side &&
                            (unsigned long long)map->width * (unsigned long long)map->height < (1ull << 32) &&
                            variant != 13;
    const bool cell_units = cell_march && map->fast_path && map->dt_cells;
    FirstLookup fl;
    fl.cells = cell_march ? (cell_units ? map->dt_cells : map->dt) : nullptr;
    fl.metres = cell_units ? 0 : 1;
    fl.res = map->resolution; fl.orig_x = map->orig_x; fl.orig_y = map->orig_y;
    fl.x_max = mv.x_max; fl.y_max = mv.y_max;
    const bool layered = map->num_layers > 1 && sim->env_layer;
    if (map->num_layers > 1 && !cell_march) return F110_ERR_INVALID;     // stacked maps need the lean march kernels
    fl.env_layer = layered ? sim->env_layer : nullptr;
    fl.layer_stride = (unsigned long long)map->width * (unsigned long long)map->height;
    fl.inv_res = 1.0 / map->resolution; fl.ox = map->orig_x * fl.inv_res; fl.oy = map->orig_y * fl.inv_res;
    fl.width = (unsigned)map->width; fl.height = (unsigned)map->height;
    fl.last = (unsigned)map->width * (unsigned)map->height - 1u;
    // the lean march kernel (march_lean.cuh): 32-beam queue items, `d > eps` == `d != 0` (every positive DT value exceeds
    // eps), fov < 2 pi (the doubled sin/cos LUT replaces the wrap), LUT indices that fit the Q16.48 fixed point
    const bool lean = queued && cell_march && item_sub == 1 && sim->march_rec && map->sincos2 && map->eps >= 0.0 &&
                      (!cell_units || map->dt_cells_pad) && (unsigned long long)NA * (unsigned long long)beams->num_beams < (1ull << 32) &&
                      (unsigned long long)(map->width + 1) * (unsigned long long)(map->height + 1) < (1ull << 32) &&
                      map->dt_min_positive > map->eps && beams->fov > 0.0 && beams->fov < 6.283185307179586 &&
                      beams->theta_index_increment > 0.0 && map->theta_dis < 32768 &&
                      variant != 1 && variant != 6;
    // the TMA-tile kernel (march_tile.cuh; variants 30 / 31): single cell-unit map with the padded code table
    const int tile_sz = (variant == 31) ? 160 : 128;
    const bool tile = lean && (variant == 30 || variant == 31) && map->fast_path && map->dt_cells_pad && map->dt_codes_pad &&
                      map->dt_lut && !(map->num_layers > 1) && map->codes_pitch >= (unsigned)tile_sz && map->codes_pitch % 16 == 0 &&
                      map->height + 1 >= tile_sz && (unsigned long long)NA * (unsigned long long)sim->march_ipa < (1ull << 24);
    if (tile) order_blocks = dyn_blocks;
    fl.agent_queue = tile ? 1 : 0;
    fl.rec = lean ? reinterpret_cast<double2 *>(sim->march_rec) : nullptr;
    fl.side_max = beams->side_max > 0.0 ? beams->side_max : INFINITY;
    fl.ttc_margin = sim->ttc_thresh * 1.000001;
    fl.rec_layer_stride = cell_units ? (unsigned long long)(map->width + 1) * (unsigned long long)(map->height + 1) : fl.layer_stride;
    k_dynamics<<<dyn_blocks + order_blocks, 128, 0, st>>>(*sim, actions, beams->fov, (double)map->theta_dis, dyn_blocks, fl);
    LAUNCH_CHECK("k_dynamics");
    if (ev) CUDA_TRY(cudaEventRecord(ev[1], st));

    if (cell_march) {
        MarchK k;
        const bool coded = cell_units && !layered && map->dt_codes && map->dt_lut && variant == 6;   // measured: the fp64 table wins once issue-bound
        k.codes = map->dt_codes; k.lut = map->dt_lut; k.cells = map->dt_cells;
        k.sincos = reinterpret_cast<const double2 *>(map->sincos);
        k.cos_side = reinterpret_cast<const double2 *>(beams->cos_side);
        k.scan_pose = reinterpret_cast<const double2 *>(sim->scan_pose);
        k.vel = sim->state + (size_t)3 * NA;
        k.out = sim->scans; k.wall_flag = sim->wall_flag;
        k.lookup_counter = sim->lookup_counter; k.tick_counter = sim->tick_counter;
        k.inv_res = 1.0 / map->resolution; k.res = map->resolution;
        k.ox = map->orig_x * k.inv_res; k.oy = map->orig_y * k.inv_res;
        k.eps = map->eps * k.inv_res; k.tmax = map->max_range * k.inv_res;
        k.inc = beams->theta_index_increment; k.theta_dis_f = (double)map->theta_dis;
        k.ti_guard = 4.0 * ((double)beams->num_beams * 1.14e-13 + 1e-12);
        k.ttc_thresh = sim->ttc_thresh; k.ttc_margin = sim->ttc_thresh * 1.000001;
        k.noise_std = sim->noise_std; k.noise_seed = sim->noise_seed;
        k.width = (unsigned)map->width; k.height = (unsigned)map->height;
        k.last = (unsigned)map->width * (unsigned)map->height - 1u;
        k.B = beams->num_beams;
        k.env_layer = layered ? sim->env_layer : nullptr;
        k.layer_stride = fl.layer_stride; k.num_agents = (unsigned)sim->num_agents;
        k.trace = g_trace;
        k.dt = map->dt; k.orig_x = map->orig_x; k.orig_y = map->orig_y; k.x_max = mv.x_max; k.y_max = mv.y_max;
        k.dt_oob = map->dt_oob; k.eps_m = map->eps; k.max_range = map->max_range;
        const int bpa = (beams->num_beams + 63) / 64;
        if (bpa > 65000) return F110_ERR_INVALID;
        const bool noise = sim->noise_std > 0.0, count = sim->lookup_counter != nullptr;
        MarchQueue mq = {};
        if (queued) {
            mq.cost = sim->march_cost; mq.order = sim->march_order; mq.count = sim->march_count;
            mq.ipa = (unsigned)sim->march_ipa; mq.items = (unsigned)NA * mq.ipa;
            if (g_chunk < 0) { const char *e = getenv("F110_MARCH_CHUNK"); g_chunk = e ? atoi(e) : 3; if (g_chunk < 0 || g_chunk > 6) g_chunk = 3; }
            mq.chunk_shift = (unsigned)g_chunk;
            mq.claim = sim->march_count + 3;
            {   // dynamic tail of the queue (k_march_lean<DYN>): g_dyn_pct % of every block's share is dealt statically
                const unsigned runs = (mq.items + (1u << mq.chunk_shift) - 1u) >> mq.chunk_shift;
                // (blocks of the lean launch: 2 per SM when the big shape is chosen -- same rule as launch_lean)
                const bool big_blocks = (variant == 42);      // the dynamic default (variants 0 / 40 / 41) runs 4 x 512 threads per SM
                const unsigned blocks = (unsigned)num_sms() * (big_blocks ? 2u : (variant == 41 || variant == 57 || variant == 58) ? 3u : 4u);
                mq.dyn_ahead = (unsigned)g_dyn_ahead;
                mq.static_runs = (unsigned)((unsigned long long)runs * (unsigned)g_dyn_pct / 100ull / blocks);
                // entries per ticket by queue class (k_march_lean<IPT = 0>)
                unsigned sh[4];
                // (at least two tickets per run: with one, the 16 warps of a block could hold tickets of 16 runs at once and
                // the claim for run r + 16 could overwrite the ring slot of run r before it is read)
                const unsigned sh_max = mq.chunk_shift > 0u ? mq.chunk_shift - 1u : 0u;
                // queue entries per warp of the launch: one entry per ticket for the very heavy runs, four for the light ones, and
                // for the heavy runs two on a short queue, four on a longer one (cfg2: 68.3 us with 0:1:2, 69.8 with 0:2:2;
                // n12288a1 and cfg2x2: 155.9 / 112.0 and 155.1 / 111.7; profiles/r2/ab_march_23_*.jsonl)
                const unsigned per_warp = mq.items / (blocks * 16u);
                const int dflt[4] = {0, per_warp >= 27u ? 2 : 1, 2, 255};
                for (int z = 0; z < 4; z++) {
                    const int want = g_ipt[z] < 0 ? dflt[z] : g_ipt[z];
                    sh[z] = (z == 3 && want == 255) ? 255u : std::min((unsigned)want, sh_max);
                }
                mq.uniform_ipt4 = (g_ipt[0] >= 0 || g_ipt[1] >= 0 || g_ipt[2] >= 0 || mq.chunk_shift < 3u) ? 0u : per_warp >= 72u ? 4u : per_warp >= 27u ? 2u : 0u;
                mq.ipt_shifts = sh[0] | (sh[1] << 8) | (sh[2] << 16) | (sh[3] << 24);
            }
        }
        if (lean) {
            LeanK q;
            q.table = cell_units ? map->dt_cells_pad : map->dt;
            q.codes = map->dt_codes_pad; q.lut = map->dt_lut;
            q.sincos2 = reinterpret_cast<const double2 *>(map->sincos2);
            q.cos_side = k.cos_side;
            q.rec = reinterpret_cast<const double2 *>(sim->march_rec);
            q.out = sim->scans; q.wall_flag = sim->wall_flag;
            q.lookup_counter = sim->lookup_counter; q.tick_counter = sim->tick_counter;
            q.res = map->resolution; q.inv_res = 1.0 / map->resolution;
            if (cell_units) { q.ox = k.ox; q.oy = k.oy; q.tmax = k.tmax; }
            else { q.ox = map->orig_x; q.oy = map->orig_y; q.tmax = map->max_range; }
            q.x_max = mv.x_max; q.y_max = mv.y_max;
            q.ttc_thresh = k.ttc_thresh; q.ttc_margin = k.ttc_margin; q.noise_std = k.noise_std; q.noise_seed = k.noise_seed;
            q.inc = k.inc; q.theta_dis_f = k.theta_dis_f;
            q.inc_fx = (unsigned long long)(beams->theta_index_increment * 281474976710656.0 + 0.5);
            // the fixed-point index is within B * 2^-49 + 2^-48 of the real closed form, which is within B * 1.14e-13 of the
            // reference's sequential sum (lidar.cuh): replay when the fraction is closer than that (x4) to an integer
            const double guard = 4.0 * ((double)beams->num_beams * 1.2e-13 + 1e-12);
            q.guard32 = (unsigned)(guard * 4294967296.0) + 2u;
            q.width = k.width; q.height = k.height; q.last = k.last; q.B = k.B;
            q.layer_stride = fl.layer_stride; q.layer_stride_lean = fl.rec_layer_stride;
            q.dt = map->dt; q.orig_x = map->orig_x; q.orig_y = map->orig_y; q.dt_oob_unused = 0.0; q.eps_m = map->eps;
            q.max_range = map->max_range;
            q.codes_pitch = map->codes_pitch;
            const bool lcoded = cell_units && !layered && map->dt_codes_pad && map->dt_lut && map->codes_pitch > (unsigned)map->width &&
                                (variant == 20 || variant == 22);
            const bool occ3 = (variant == 21 || variant == 22 || variant == 41);
            if (tile) {
                TileK t;
                t.l = q;
                t.order = sim->march_order; t.count = sim->march_count; t.claim = sim->march_count + 3;
                t.cost = sim->march_cost; t.agents = (unsigned)NA; t.ipa = (unsigned)sim->march_ipa;
                t.ipa_magic = (unsigned)(4294967296ull / (unsigned long long)sim->march_ipa) + 1u;
                t.codes_pitch = map->codes_pitch;
                t.c_max = (int)map->codes_pitch - tile_sz; t.r_max = map->height + 1 - tile_sz;
                t.tile_counter = g_tile_counter;
                if ((rc = launch_tile(t, map, tile_sz, (unsigned)num_sms(), noise, count, st))) return rc;
            } else
            launch_lean(q, mq, (unsigned)num_sms(), cell_units, lcoded, occ3, layered, noise, count,
                        /* dynamic queue tail: */ (variant == 0 || variant == 40 || variant == 41 || variant == 42 || variant == 43 || variant == 45 || variant == 57 || variant == 58 || (variant >= 81 && variant <= 86)) && !layered &&
                            mq.static_runs >= mq.dyn_ahead, st);
        } else if (queued) {
            const unsigned blocks = (unsigned)num_sms() * 4u;
            if (!cell_units) launch_persistent<512, 1, false>(k, mq, blocks, coded, noise, count, st);
            else if (item_sub == 2) launch_persistent<512, 2, true>(k, mq, blocks, coded, noise, count, st);
            else launch_persistent<512, 1, true>(k, mq, blocks, coded, noise, count, st);
        } else {
            const dim3 grid((unsigned)NA, (unsigned)bpa);
            if (!cell_units) launch_march<32, false>(k, grid, coded, noise, count, st);
            else if (variant == 9) launch_march<24, true>(k, grid, coded, noise, count, st);
            else launch_march<32, true>(k, grid, coded, noise, count, st);
        }
        LAUNCH_CHECK("k_march");
        goto marched;
    }
    {
    MarchArgs g;
    g.scan_pose = sim->scan_pose;
    g.vel = sim->state + (size_t)3 * NA;
    g.out_f32 = sim->scans;
    g.out_f64 = nullptr;
    g.wall_flag = sim->wall_flag;
    g.lookup_counter = sim->lookup_counter;
    g.tick_counter = sim->tick_counter;
    g.ttc_thresh = sim->ttc_thresh;
    g.noise_std = sim->noise_std;
    g.noise_seed = sim->noise_seed;
    g.total = (long long)NA * beams->num_beams;
    if ((rc = launch_raymarch(mv, bv, g, map->fast_path != 0, false, st))) return rc;
    }
marched:
    if (ev) CUDA_TRY(cudaEventRecord(ev[2], st));

    // largest value a scan entry can hold: the max_range clamp plus 8 sigma of the optional noise
    const double max_scan = map->max_range + 8.0 * (sim->noise_std > 0.0 ? sim->noise_std : 0.0) + 1e-3;
    // k_tail2 (2 <= A <= 4): cfg3 tail 79 -> 60 us, tick 518 -> 486 us; cfg2x2 28.5 -> 22.6 us once its blocks are small enough to
    // fill the GPU (profiles/r2/ab_march_16..18_*.jsonl)
    if (sim->num_agents >= 2 && sim->num_agents <= 4 && g_tail2) {
        // two-phase tail: ~64 agents per block (thread per (ego, opponent) pair for the scalar work, warp per ego for the beams);
        // f110_step (no lap logic, no auto-reset) runs the same kernel with the env-level phase switched off
        // up to 64 agents per block, fewer when that would leave SMs without a block (cfg2x2: 4096 envs / 32 = 128 blocks lost
        // 4 us against 8 envs per block)
        int epb = g_tail2_forced ? max(1, g_tail2_agents / sim->num_agents) : max(1, min(g_tail2_agents / sim->num_agents, sim->num_envs / (4 * num_sms())));
        AutoResetArgs no_ar;
        no_ar.start_poses = nullptr; no_ar.num_start = 0; no_ar.pose_gap = 0; no_ar.seed = 0; no_ar.tick_host = 0;
        const bool fused = tail && tail->fused;
        // big blocks (>= 48 agents) run 256 threads, small ones 128 (measured: 256:64 best at cfg3, 128:12 at cfg2x2)
        int t2 = (g_tail2_threads != F110_TAIL2_THREADS) ? g_tail2_threads : (epb * sim->num_agents >= 48 ? 256 : 128);
        if (!g_tail2_forced && g_tail2_threads == F110_TAIL2_THREADS) {
            // Whole waves.  With 80 registers an SM holds six 128-thread blocks (three of 256 threads); a grid of 1.37 waves (cfg3:
            // 607 blocks of 27 envs, 256 threads, on 444 slots) leaves the GPU two-thirds empty for the second half of the kernel:
            // 59.4 us against 46.8 for 863 blocks of 19 envs on the 888 slots of 128-thread blocks, 46.5 for 443 blocks of 37 envs
            // at 256 threads (profiles/r2/ab_march_31_tail2_waves.jsonl).  So: 128-thread blocks of up to 47 agents, and as many
            // envs per block as fill a whole number of waves.
            static int per_sm = 0;                          // resident 128-thread blocks per SM
            if (per_sm == 0) {
                const size_t sm0 = (size_t)(47 / sim->num_agents) * sim->num_agents * (sim->num_agents - 1) * sizeof(TailTask);
                if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_tail2, 128, sm0) != cudaSuccess || per_sm < 1) { per_sm = -1; cudaGetLastError(); }
            }
            if (per_sm > 0) {
                const long long cap = (long long)per_sm * num_sms();
                const long long emax = max(1, 47 / sim->num_agents);
                const long long waves = (sim->num_envs + cap * emax - 1) / (cap * emax);
                epb = (int)((sim->num_envs + waves * cap - 1) / (waves * cap));
                t2 = 128;
            }
        }
        const size_t smem = (size_t)epb * sim->num_agents * (sim->num_agents - 1) * sizeof(TailTask);
        launch_k(k_tail2, dim3((sim->num_envs + epb - 1) / epb), dim3(t2), smem, st, g_pdl_this_step && lean, *sim, bv,
                 fused ? (int)tail->env_level : 0, fused ? tail->ar : no_ar, max_scan, epb);
        LAUNCH_CHECK("k_tail2");
    } else if (tail && tail->fused && sim->num_agents <= 32) {
        // whole envs per block, ~4 warps per block: A = 1 -> 4 envs, A = 2 -> 2 envs, A >= 4 -> 1 env
        const int epb = sim->num_agents >= 4 ? 1 : 4 / sim->num_agents;
        const int threads = 32 * sim->num_agents * epb;
        const dim3 tgrid((sim->num_envs + epb - 1) / epb);
        const bool tpdl = g_pdl_this_step && lean;
        // register budget of the 128-thread flavour (A <= 4): 4 blocks/SM = 128 registers (no spills), 5 = 96, 8 = 64
        if (threads <= 128 && g_tail_minb == 4)
            launch_k(k_tail<128, 4>, tgrid, dim3(threads), 0, st, tpdl, *sim, bv, (int)tail->env_level, tail->ar, max_scan, epb);
        else if (threads <= 128 && g_tail_minb == 5)
            launch_k(k_tail<128, 5>, tgrid, dim3(threads), 0, st, tpdl, *sim, bv, (int)tail->env_level, tail->ar, max_scan, epb);
        else if (threads <= 128)
            launch_k(k_tail<128, 8>, tgrid, dim3(threads), 0, st, tpdl, *sim, bv, (int)tail->env_level, tail->ar, max_scan, epb);
        else
            launch_k(k_tail<1024, 1>, dim3((sim->num_envs + epb - 1) / epb), dim3(threads), 0, st, g_pdl_this_step && lean, *sim, bv,
                     (int)tail->env_level, tail->ar, max_scan, epb);
        LAUNCH_CHECK("k_tail");
    } else {
        launch_k(k_finalize, dim3((NA * 32 + 127) / 128), dim3(128), 0, st, g_pdl_this_step && lean, *sim, bv, max_scan);
        LAUNCH_CHECK("k_finalize");
        if (tail && tail->fused) {     // more than 32 agents per env: same semantics with separate launches
            if (tail->env_level) { k_env_post_step<<<(sim->num_envs + 127) / 128, 128, 0, st>>>(*sim); LAUNCH_CHECK("k_env_post_step"); }
            if (tail->ar.start_poses) { k_autoreset<<<(sim->num_envs + 127) / 128, 128, 0, st>>>(*sim, tail->ar); LAUNCH_CHECK("k_autoreset"); }
        }
    }
    if (ev) CUDA_TRY(cudaEventRecord(ev[3], st));
    return F110_OK;
}

int f110_step(const f110_sim *sim, const f110_map *map, const f110_beams *beams, const double *actions,
              void *stream) {
    return step_impl(sim, map, beams, actions, (cudaStream_t)stream, nullptr);
}

int f110_step_profile(const f110_sim *sim, const f110_map *map, const f110_beams *beams, const double *actions,
                      float *kernel_ms /* host [3] */, void *stream) {
    if (!kernel_ms) return F110_ERR_INVALID;
    cudaEvent_t ev[4];
    for (int i = 0; i < 4; i++) CUDA_TRY(cudaEventCreate(&ev[i]));
    int rc = step_impl(sim, map, beams, actions, (cudaStream_t)stream, ev);
    if (rc == F110_OK) {
        cudaError_t e = cudaEventSynchronize(ev[3]);
        if (e != cudaSuccess) rc = cuda_fail(e, "cudaEventSynchronize");
        for (int i = 0; i < 3 && rc == F110_OK; i++) {
            e = cudaEventElapsedTime(&kernel_ms[i], ev[i], ev[i + 1]);
            if (e != cudaSuccess) rc = cuda_fail(e, "cudaEventElapsedTime");
        }
    }
    for (int i = 0; i < 4; i++) cudaEventDestroy(ev[i]);
    return rc;
}

int f110_reset(const f110_sim *sim, const double *poses, const uint8_t *env_mask, void *stream) {
    int rc;
    if ((rc = check_sim(sim))) return rc;
    if (!poses) return F110_ERR_INVALID;
    const int NA = sim->num_envs * sim->num_agents;
    k_reset<<<(NA + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*sim, poses, env_mask);
    LAUNCH_CHECK("k_reset");
    return F110_OK;
}

static int check_env_arrays(const f110_sim *s) {
    if (!s->current_time || !s->lap_times || !s->lap_counts || !s->toggle_list || !s->near_starts ||
        !s->start_xs || !s->start_ys || !s->start_thetas || !s->start_rot || !s->done)
        return F110_ERR_INVALID;
    if (s->ego_idx < 0 || s->ego_idx >= s->num_agents) return F110_ERR_AGENT_INDEX;
    return F110_OK;
}

int f110_env_reset(const f110_sim *sim, const double *poses, const uint8_t *env_mask, void *stream) {
    int rc;
    if ((rc = check_sim(sim)) || (rc = check_env_arrays(sim))) return rc;
    if (!poses) return F110_ERR_INVALID;
    k_env_reset<<<(sim->num_envs + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*sim, poses, env_mask);
    LAUNCH_CHECK("k_env_reset");
    return F110_OK;
}

int f110_env_post_step(const f110_sim *sim, void *stream) {
    int rc;
    if ((rc = check_sim(sim)) || (rc = check_env_arrays(sim))) return rc;
    k_env_post_step<<<(sim->num_envs + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*sim);
    LAUNCH_CHECK("k_env_post_step");
    return F110_OK;
}

int f110_autoreset(const f110_sim *sim, const double *start_poses, int32_t num_start, int32_t pose_gap,
                   uint64_t seed, uint64_t tick, void *stream) {
    int rc;
    if ((rc = check_sim(sim))) return rc;
    if (!start_poses || num_start <= 0) return F110_ERR_INVALID;
    if (sim->ego_idx < 0 || sim->ego_idx >= sim->num_agents) return F110_ERR_AGENT_INDEX;
    if (sim->num_agents > 32) return F110_ERR_INVALID;      // the device-side auto-reset stages at most 32 start poses per env
    AutoResetArgs ar;
    ar.start_poses = start_poses; ar.num_start = num_start; ar.pose_gap = pose_gap; ar.seed = seed; ar.tick_host = tick;
    k_autoreset<<<(sim->num_envs + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*sim, ar);
    LAUNCH_CHECK("k_autoreset");
    return F110_OK;
}

int f110_tick(const f110_sim *sim, const f110_map *map, const f110_beams *beams, const double *actions,
              int32_t env_level, const double *start_poses, int32_t num_start, int32_t pose_gap, uint64_t seed,
              void *stream) {
    int rc;
    if ((rc = check_sim(sim))) return rc;
    if (env_level && (rc = check_env_arrays(sim))) return rc;
    if (start_poses && (num_start <= 0 || sim->ego_idx < 0 || sim->ego_idx >= sim->num_agents || sim->num_agents > 32))
        return F110_ERR_INVALID;
    TailOpts t;
    t.fused = true; t.env_level = env_level;
    t.ar.start_poses = start_poses; t.ar.num_start = num_start; t.ar.pose_gap = pose_gap; t.ar.seed = seed; t.ar.tick_host = 0;
    return step_impl(sim, map, beams, actions, (cudaStream_t)stream, nullptr, &t);
}

int f110_step_host(const f110_sim *sim, const f110_map *map, const f110_beams *beams, const double *actions_host,
                   double *actions_dev_scratch, const f110_host_obs *out, void *stream) {
    int rc;
    if ((rc = check_sim(sim))) return rc;
    if (!actions_host || !actions_dev_scratch || !out) return F110_ERR_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t NA = (size_t)sim->num_envs * sim->num_agents;
    CUDA_TRY(cudaMemcpyAsync(actions_dev_scratch, actions_host, NA * 2 * sizeof(double), cudaMemcpyHostToDevice, st));
    const bool env_level = sim->current_time && sim->done;
    if (env_level && (rc = check_env_arrays(sim))) return rc;
    TailOpts t;
    t.fused = true; t.env_level = env_level ? 1 : 0;
    t.ar.start_poses = nullptr; t.ar.num_start = 0; t.ar.pose_gap = 0; t.ar.seed = 0; t.ar.tick_host = 0;
    if ((rc = step_impl(sim, map, beams, actions_dev_scratch, st, nullptr, &t))) return rc;
    if (out->scans)
        CUDA_TRY(cudaMemcpyAsync(out->scans, sim->scans, NA * beams->num_beams * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (out->state)
        CUDA_TRY(cudaMemcpyAsync(out->state, sim->state, NA * 7 * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (out->collisions)
        CUDA_TRY(cudaMemcpyAsync(out->collisions, sim->collisions, NA * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (env_level) {
        if (out->done)
            CUDA_TRY(cudaMemcpyAsync(out->done, sim->done, (size_t)sim->num_envs, cudaMemcpyDeviceToHost, st));
        if (out->lap_times)
            CUDA_TRY(cudaMemcpyAsync(out->lap_times, sim->lap_times, NA * sizeof(double), cudaMemcpyDeviceToHost, st));
        if (out->lap_counts)
            CUDA_TRY(cudaMemcpyAsync(out->lap_counts, sim->lap_counts, NA * sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    CUDA_TRY(cudaStreamSynchronize(st));
    return F110_OK;
}

int f110_step_host_async(const f110_sim *sim, const f110_map *map, const f110_beams *beams,
                         const double *actions_host, double *actions_dev_scratch, const f110_host_obs *stage,
                         const f110_host_obs *out, void *compute_stream, void *copy_stream, void *ev_tick_done,
                         void *ev_copy_done) {
    int rc;
    if ((rc = check_sim(sim))) return rc;
    if (!actions_host || !actions_dev_scratch || !stage || !out || !ev_tick_done || !ev_copy_done) return F110_ERR_INVALID;
    cudaStream_t cs = (cudaStream_t)compute_stream, ps = (cudaStream_t)copy_stream;
    cudaEvent_t e_tick = (cudaEvent_t)ev_tick_done, e_copy = (cudaEvent_t)ev_copy_done;
    const size_t NA = (size_t)sim->num_envs * sim->num_agents;
    const bool env_level = sim->current_time && sim->done;
    if (env_level && (rc = check_env_arrays(sim))) return rc;
    CUDA_TRY(cudaMemcpyAsync(actions_dev_scratch, actions_host, NA * 2 * sizeof(double), cudaMemcpyHostToDevice, cs));
    TailOpts t;
    t.fused = true; t.env_level = env_level ? 1 : 0;
    t.ar.start_poses = nullptr; t.ar.num_start = 0; t.ar.pose_gap = 0; t.ar.seed = 0; t.ar.tick_host = 0;
    if ((rc = step_impl(sim, map, beams, actions_dev_scratch, cs, nullptr, &t))) return rc;
    // the staging buffers may still be draining to the host from their previous use
    CUDA_TRY(cudaStreamWaitEvent(cs, e_copy, 0));
    struct Part { void *dst_dev, *dst_host; const void *src; size_t bytes; };
    const Part parts[6] = {
        { stage->scans, out->scans, sim->scans, NA * beams->num_beams * sizeof(float) },
        { stage->state, out->state, sim->state, NA * 7 * sizeof(double) },
        { stage->collisions, out->collisions, sim->collisions, NA * sizeof(double) },
        { stage->done, out->done, env_level ? sim->done : nullptr, (size_t)sim->num_envs },
        { stage->lap_times, out->lap_times, env_level ? sim->lap_times : nullptr, NA * sizeof(double) },
        { stage->lap_counts, out->lap_counts, env_level ? sim->lap_counts : nullptr, NA * sizeof(double) },
    };
    for (int i = 0; i < 6; i++)
        if (parts[i].dst_dev && parts[i].dst_host && parts[i].src)
            CUDA_TRY(cudaMemcpyAsync(parts[i].dst_dev, parts[i].src, parts[i].bytes, cudaMemcpyDeviceToDevice, cs));
    // narrow scan block: the snapshot IS the packing (3 bytes per beam cross PCIe instead of 4)
    const bool packed = !stage->scans && !out->scans && stage->scans_u24 && out->scans_u24;
    if (packed && (rc = f110_pack_scans_u24(sim->scans, (int64_t)(NA * beams->num_beams), stage->scans_u24, cs))) return rc;
    CUDA_TRY(cudaEventRecord(e_tick, cs));
    CUDA_TRY(cudaStreamWaitEvent(ps, e_tick, 0));
    for (int i = 0; i < 6; i++)
        if (parts[i].dst_dev && parts[i].dst_host && parts[i].src)
            CUDA_TRY(cudaMemcpyAsync(parts[i].dst_host, parts[i].dst_dev, parts[i].bytes, cudaMemcpyDeviceToHost, ps));
    if (packed)
        CUDA_TRY(cudaMemcpyAsync(out->scans_u24, stage->scans_u24, NA * beams->num_beams * 3, cudaMemcpyDeviceToHost, ps));
    CUDA_TRY(cudaEventRecord(e_copy, ps));
    return F110_OK;
}

int f110_scan(const f110_map *map, const f110_beams *beams, const double *poses, int32_t M, float *out_f32,
              double *out_f64, unsigned long long *lookup_counter, void *stream) {
    int rc;
    if ((rc = check_map(map)) || (rc = check_beams(beams))) return rc;
    if (!poses || M <= 0 || (!out_f32 && !out_f64)) return F110_ERR_INVALID;
    MarchArgs g;
    memset(&g, 0, sizeof(g));
    g.scan_pose = poses;
    g.out_f32 = out_f32;
    g.out_f64 = out_f64;
    g.lookup_counter = lookup_counter;
    g.total = (long long)M * beams->num_beams;
    return launch_raymarch(make_view(map), make_view(beams), g, map->fast_path != 0, true, (cudaStream_t)stream);
}

int f110_vehicle_dynamics_st(const double *x, const double *u, const double *params, int32_t M, double *f, void *stream) {
    if (!x || !u || !params || !f || M <= 0) return F110_ERR_INVALID;
    k_rhs<<<(M + 127) / 128, 128, 0, (cudaStream_t)stream>>>(x, u, params, M, f);
    LAUNCH_CHECK("k_rhs");
    return F110_OK;
}

int f110_vehicle_dynamics_ks(const double *x, const double *u, const double *params, int32_t M, double *f, void *stream) {
    if (!x || !u || !params || !f || M <= 0) return F110_ERR_INVALID;
    k_rhs_ks<<<(M + 127) / 128, 128, 0, (cudaStream_t)stream>>>(x, u, params, M, f);
    LAUNCH_CHECK("k_rhs_ks");
    return F110_OK;
}

int f110_pid(const double *in, const double *params, int32_t M, double *out, void *stream) {
    if (!in || !params || !out || M <= 0) return F110_ERR_INVALID;
    k_pid<<<(M + 127) / 128, 128, 0, (cudaStream_t)stream>>>(in, params, M, out);
    LAUNCH_CHECK("k_pid");
    return F110_OK;
}

int f110_get_vertices(const double *poses, double length, double width, int32_t M, double *out, void *stream) {
    if (!poses || !out || M <= 0) return F110_ERR_INVALID;
    k_vertices<<<(M + 127) / 128, 128, 0, (cudaStream_t)stream>>>(poses, length, width, M, out);
    LAUNCH_CHECK("k_vertices");
    return F110_OK;
}

int f110_collision(const double *va, const double *vb, int32_t M, int32_t *out, void *stream) {
    if (!va || !vb || !out || M <= 0) return F110_ERR_INVALID;
    k_gjk<<<(M + 127) / 128, 128, 0, (cudaStream_t)stream>>>(va, vb, M, out);
    LAUNCH_CHECK("k_gjk");
    return F110_OK;
}

int f110_collision_multiple(const double *verts, int32_t M, int32_t n, double *collisions, double *collision_idx,
                            void *stream) {
    if (!verts || !collisions || !collision_idx || M <= 0 || n <= 0) return F110_ERR_INVALID;
    k_gjk_multiple<<<(M + 63) / 64, 64, 0, (cudaStream_t)stream>>>(verts, M, n, collisions, collision_idx);
    LAUNCH_CHECK("k_gjk_multiple");
    return F110_OK;
}

int f110_check_ttc(const f110_beams *beams, const double *scans, const double *vel, double ttc_thresh, int32_t M,
                   int32_t *out, void *stream) {
    int rc;
    if ((rc = check_beams(beams))) return rc;
    if (!scans || !vel || !out || M <= 0) return F110_ERR_INVALID;
    k_check_ttc<<<((long long)M * 32 + 127) / 128, 128, 0, (cudaStream_t)stream>>>(make_view(beams), scans, vel,
                                                                                   ttc_thresh, M, out);
    LAUNCH_CHECK("k_check_ttc");
    return F110_OK;
}

int f110_ray_cast(const f110_beams *beams, const double *poses, const double *opp_vertices, int32_t M, float *scans,
                  int32_t *window, void *stream) {
    int rc;
    if ((rc = check_beams(beams))) return rc;
    if (!poses || !opp_vertices || !scans || M <= 0) return F110_ERR_INVALID;
    k_ray_cast<<<((long long)M * 32 + 127) / 128, 128, 0, (cudaStream_t)stream>>>(make_view(beams), poses, opp_vertices,
                                                                                  M, scans, window);
    LAUNCH_CHECK("k_ray_cast");
    return F110_OK;
}

int f110_pure_pursuit(const double *wx, const double *wy, const double *wv, int32_t num_waypoints, const double *pose_x,
                      const double *pose_y, const double *pose_theta, int32_t M, double lookahead_distance, double vgain,
                      double wheelbase, double max_reacquire, double *actions_out, void *stream) {
    if (!wx || !wy || !wv || num_waypoints < 2 || !pose_x || !pose_y || !pose_theta || M <= 0 || !actions_out)
        return F110_ERR_INVALID;
    k_pure_pursuit<<<((long long)M * 32 + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
        wx, wy, wv, num_waypoints, nullptr, nullptr, pose_x, pose_y, pose_theta, M, lookahead_distance, vgain, wheelbase,
        max_reacquire, actions_out);
    LAUNCH_CHECK("k_pure_pursuit");
    return F110_OK;
}

int f110_pure_pursuit_tables(const double *wx, const double *wy, const double *wv, const int32_t *table_start,
                             int32_t num_tables, const int32_t *pose_table, const double *pose_x, const double *pose_y,
                             const double *pose_theta, int32_t M, double lookahead_distance, double vgain, double wheelbase,
                             double max_reacquire, double *actions_out, void *stream) {
    if (!wx || !wy || !wv || !table_start || num_tables <= 0 || !pose_table || !pose_x || !pose_y || !pose_theta || M <= 0 ||
        !actions_out)
        return F110_ERR_INVALID;
    k_pure_pursuit<<<((long long)M * 32 + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
        wx, wy, wv, 0, table_start, pose_table, pose_x, pose_y, pose_theta, M, lookahead_distance, vgain, wheelbase,
        max_reacquire, actions_out);
    LAUNCH_CHECK("k_pure_pursuit");
    return F110_OK;
}

int f110_edt(const uint8_t *occupied, int32_t height, int32_t width, double resolution, int32_t *scratch, double *dt_out,
             int64_t *k_out, void *stream) {
    if (!occupied || !scratch || !dt_out || height <= 0 || width <= 0 || !(resolution > 0)) return F110_ERR_INVALID;
    if ((size_t)width * sizeof(int32_t) > 200 * 1024) return F110_ERR_INVALID;      // one row of g must fit in shared memory
    cudaStream_t st = (cudaStream_t)stream;
    k_edt_columns<<<(width + 127) / 128, 128, 0, st>>>(occupied, height, width, scratch);
    LAUNCH_CHECK("k_edt_columns");
    const size_t smem = (size_t)width * sizeof(int32_t);
    if (smem > 48 * 1024)
        CUDA_TRY(cudaFuncSetAttribute(k_edt_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_edt_rows<<<height, 256, smem, st>>>(scratch, height, width, resolution, dt_out, k_out);
    LAUNCH_CHECK("k_edt_rows");
    return F110_OK;
}

int f110_rasterize_track(const double *segments, int32_t num_segments, double wall_inner, double wall_outer, int32_t height,
                          int32_t width, uint8_t *occupied, double *dist2_out, void *stream) {
    if (!segments || !occupied || num_segments <= 0 || height <= 0 || width <= 0 || !(wall_inner >= 0) ||
        !(wall_outer >= wall_inner))
        return F110_ERR_INVALID;
    const size_t smem = (size_t)num_segments * 5 * sizeof(double);
    if (smem > 200 * 1024) return F110_ERR_INVALID;
    if (smem > 48 * 1024)
        CUDA_TRY(cudaFuncSetAttribute(k_rasterize_track, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const dim3 block(32, 8), grid((width + 31) / 32, (height + 7) / 8);
    k_rasterize_track<<<grid, block, smem, (cudaStream_t)stream>>>(segments, num_segments, wall_inner * wall_inner,
                                                                    wall_outer * wall_outer, height, width, occupied, dist2_out);
    LAUNCH_CHECK("k_rasterize_track");
    return F110_OK;
}

int f110_pack_scans_u24(const float *scans, int64_t count, uint8_t *out, void *stream) {
    if (!scans || !out || count <= 0) return F110_ERR_INVALID;
    const long long groups = (count + 3) / 4;
    k_pack_u24<<<(unsigned)((groups + 255) / 256), 256, 0, (cudaStream_t)stream>>>(scans, (long long)count, out);
    LAUNCH_CHECK("k_pack_u24");
    return F110_OK;
}

int f110_scan_noise(float *scans, int64_t count, double std_dev, uint64_t seed, uint64_t offset, void *stream) {
    if (!scans || count <= 0) return F110_ERR_INVALID;
    k_scan_noise<<<(unsigned)((count + 255) / 256), 256, 0, (cudaStream_t)stream>>>(scans, count, std_dev, seed, offset);
    LAUNCH_CHECK("k_scan_noise");
    return F110_OK;
}

int f110_render(const f110_sim *sim, const f110_map *map, const f110_beams *beams, const f110_view *view,
                const int32_t *viewers, int32_t num_frames, uint8_t *out, double *camera_out, void *stream) {
    if (!sim || !view || !out || ((uintptr_t)out & 3)) return F110_ERR_INVALID;
    if (sim->num_envs <= 0 || sim->num_agents <= 0 || !sim->state || !(sim->sim_length > 0) || !(sim->sim_width > 0))
        return F110_ERR_INVALID;
    if ((long long)sim->num_envs * sim->num_agents > 0x7FFFFFFFLL) return F110_ERR_INVALID;
    const f110_view &v = *view;
    if (v.width <= 0 || v.height <= 0 || v.width % 4 != 0 || (v.channels != 1 && v.channels != 3) ||
        (v.camera != 0 && v.camera != 1) || !(v.metres_per_pixel > 0) || !isfinite(v.metres_per_pixel) ||
        !isfinite(v.center_x) || !isfinite(v.center_y))
        return F110_ERR_INVALID;
    const long long groups = (long long)(v.width / 4) * v.height;
    if (groups > 0x7FFFFFFFLL) return F110_ERR_INVALID;
    if (num_frames <= 0 || (!viewers && num_frames != sim->num_envs)) return F110_ERR_INVALID;
    if (v.draw_scan && (check_beams(beams) || !sim->scans || !sim->scan_pose || !sim->agent_poses)) return F110_ERR_INVALID;
    if (v.num_waypoints < 0 || (v.num_waypoints > 0 && (!v.wx || !v.wy))) return F110_ERR_INVALID;
    if (v.table_start && (v.num_tables <= 0 || !v.env_table)) return F110_ERR_INVALID;
    const size_t smem = (size_t)sim->num_agents * F110_RENDER_CAR * sizeof(double);
    if (smem > 200 * 1024) return F110_ERR_INVALID;
    int rc;
    if ((rc = check_map(map))) return rc;

    RenderArgs r;
    memset(&r, 0, sizeof(r));
    r.dt = map->dt;
    r.orig_x = map->orig_x; r.orig_y = map->orig_y; r.orig_c = map->orig_c; r.orig_s = map->orig_s;
    r.resolution = map->resolution; r.inv_resolution = 1.0 / map->resolution;
    r.x_max = map->width * map->resolution;          // `width * resolution` (laser_models.py:79), as in make_view
    r.y_max = map->height * map->resolution;
    r.map_h = map->height; r.map_w = map->width;
    r.layer_stride = (unsigned long long)map->height * (unsigned long long)map->width;
    r.env_layer = (map->num_layers > 1) ? sim->env_layer : nullptr;
    r.state = sim->state;
    r.num_envs = sim->num_envs; r.num_agents = sim->num_agents; r.ego_idx = sim->ego_idx;
    r.length = sim->sim_length; r.width = sim->sim_width;
    r.W = v.width; r.H = v.height; r.channels = v.channels; r.camera = v.camera;
    r.center_x = v.center_x; r.center_y = v.center_y; r.mpp = v.metres_per_pixel;
    memcpy(r.palette, v.palette, sizeof(r.palette));
    r.viewers = viewers; r.num_frames = num_frames; r.out = out;

    cudaStream_t st = (cudaStream_t)stream;
    const unsigned fy = num_frames < 65535 ? (unsigned)num_frames : 65535u;
    const dim3 grid((unsigned)((groups + F110_RENDER_THREADS - 1) / F110_RENDER_THREADS), fy);
    // fast_path (power-of-two resolution, unrotated origin): x * (1/res) is the same number as x / res
    auto kf = map->fast_path ? k_render_frame<true> : k_render_frame<false>;
    if (smem > 48 * 1024) CUDA_TRY(cudaFuncSetAttribute(kf, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kf<<<grid, F110_RENDER_THREADS, smem, st>>>(r, camera_out);
    LAUNCH_CHECK("k_render_frame");
    if (v.draw_scan) {
        const int B = beams->num_beams;
        k_render_scan<<<dim3((B + F110_RENDER_THREADS - 1) / F110_RENDER_THREADS, fy), F110_RENDER_THREADS, 0, st>>>(
            r, sim->scans, sim->scan_pose, sim->agent_poses, beams->scan_angles, B, map->max_range);
        LAUNCH_CHECK("k_render_scan");
    }
    if (v.num_waypoints > 0) {
        k_render_waypoints<<<dim3((v.num_waypoints + F110_RENDER_THREADS - 1) / F110_RENDER_THREADS, fy), F110_RENDER_THREADS, 0,
                             st>>>(r, v.wx, v.wy, v.num_waypoints, v.table_start, v.num_tables, v.env_table);
        LAUNCH_CHECK("k_render_waypoints");
    }
    return F110_OK;
}

}  // extern "C"
