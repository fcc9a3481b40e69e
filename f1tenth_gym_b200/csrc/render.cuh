// render.cuh — headless top-down frames of the batch, straight into device memory (no window, no GL).
//
// Replaces the drawing part of the reference's rendering.py / F110Env.render for the two uses a batched gym has for it:
// rgb_array frames for videos and small per-agent bird's-eye label frames as a policy input.  Semantics (exact; the numpy
// restatement in oracle/render.py matches them bit for bit, include/f110_b200.h documents them for users):
//   pixel (r, c) centre in camera metres   u = (c + 0.5 - 0.5 W) mpp,  v = (0.5 H - r - 0.5) mpp
//   in world metres                        x = cx + (u cr - v sr),     y = cy + (u sr + v cr)
//   label  0 free / off-map, 1 wall (dt == 0 under the literal xy_2_rc of laser_models.py:55-86), 2 the viewer's car,
//          3 another car of the viewer's env, 4 a scan endpoint of the viewer, 5 a waypoint.
// A frame is computed by k_render_frame (gather: labels 0-3); the point layers are stream-ordered scatter launches after it.
#pragma once
#include <math.h>
#include <stdint.h>

#include "collision.cuh"

namespace f110 {

#define F110_RENDER_THREADS 256
#define F110_RENDER_CAR 12          // doubles per car in shared memory: 4 vertices (x, y), then lo x, hi x, lo y, hi y

struct RenderArgs {
    // map (ScanSimulator2D state)
    const double *__restrict__ dt;
    double orig_x, orig_y, orig_c, orig_s, resolution, inv_resolution, x_max, y_max;
    int32_t map_h, map_w;
    unsigned long long layer_stride;           // elements per map layer
    const int32_t *__restrict__ env_layer;     // stacked maps: layer of each env, or NULL
    // simulation
    const double *__restrict__ state;          // [7][N*A]
    int32_t num_envs, num_agents, ego_idx;
    double length, width;
    // view
    int32_t W, H, channels, camera;
    double center_x, center_y, mpp;
    uint8_t palette[8][3];
    const int32_t *__restrict__ viewers;       // [F] flat agent indices, or NULL: frame f shows env f from its ego
    int32_t num_frames;
    uint8_t *__restrict__ out;                 // [F][H][W][channels]
};

// flat agent index of frame f's viewer, or -1 when it is out of range (the frame stays all 0)
__device__ __forceinline__ int render_viewer(const RenderArgs &r, int f) {
    const int A = r.num_agents, NA = r.num_envs * r.num_agents;
    if (!r.viewers) return (r.ego_idx >= 0 && r.ego_idx < A) ? f * A + r.ego_idx : -1;
    const int a = __ldg(r.viewers + f);
    return (a >= 0 && a < NA) ? a : -1;
}

// The edge-function predicate of the spec: all four (b - a) x (p - a) >= 0 over the edges rl-rr, rr-fr, fr-fl, fl-rl.  The
// bounding-box early-out cannot change it: the box is widened by 1e-6 of the car's extent, and a point that far outside the
// box is at least that distance / sqrt(2) from the line of some edge, which is ~1e9 times what the roundings of an edge
// function can move its sign (a few ulp of |b - a| |p - a|).  A NaN coordinate fails both tests alike.
__device__ __forceinline__ bool render_in_car(const double *__restrict__ c, double px, double py) {
    if (px < c[8] || px > c[9] || py < c[10] || py > c[11]) return false;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int j = (i + 1) & 3;
        const double ax = c[2 * i], ay = c[2 * i + 1], bx = c[2 * j], by = c[2 * j + 1];
        if (!((bx - ax) * (py - ay) - (by - ay) * (px - ax) >= 0.0)) return false;
    }
    return true;
}

// label 1 test: the literal xy_2_rc (laser_models.py:55-86, dt_lookup<false> in lidar.cuh); off the map is free.  FAST (power-of-two
// resolution, unrotated origin) multiplies by 1/res, which is then the same number as the division.  An index that rounds up to
// the table's width or height is off the map too (the reference would read past its table there).
template <bool FAST>
__device__ __forceinline__ bool render_wall(const RenderArgs &r, const double *__restrict__ dt, double x, double y) {
    const double tx = x - r.orig_x, ty = y - r.orig_y;
    const double xr = tx * r.orig_c + ty * r.orig_s;
    const double yr = -tx * r.orig_s + ty * r.orig_c;
    if (!(xr >= 0 && xr < r.x_max && yr >= 0 && yr < r.y_max)) return false;    // a NaN coordinate is off the map too
    const int c = FAST ? (int)(xr * r.inv_resolution) : (int)(xr / r.resolution);
    const int row = FAST ? (int)(yr * r.inv_resolution) : (int)(yr / r.resolution);
    if (c >= r.map_w || row >= r.map_h) return false;
    return __ldg(dt + (size_t)row * (size_t)r.map_w + (size_t)c) == 0.0;
}

// The frame's camera (thread 0, also to camera_out) and the A cars of the viewer's env with their widened boxes, into shared memory.
// Out of line, with scalar arguments: fp64 sin / cos carry a rarely taken argument-reduction call that would otherwise cost the
// pixel loop registers.
__device__ __noinline__ void render_prepare(const double *__restrict__ state, int num_envs, int A, int a, int camera, double center_x,
                                            double center_y, bool cars, double length, double width, double *s_cam,
                                            double *s_car, double *__restrict__ camera_out) {
    const size_t NA = (size_t)num_envs * (size_t)A;
    if (threadIdx.x == 0) {
        if (a < 0) {
            s_cam[0] = s_cam[1] = s_cam[2] = s_cam[3] = 0.0;
        } else if (camera == 0) {
            s_cam[0] = center_x; s_cam[1] = center_y; s_cam[2] = 1.0; s_cam[3] = 0.0;
        } else {
            const double yaw = state[4 * NA + a];
            s_cam[0] = state[a]; s_cam[1] = state[NA + a];
            s_cam[2] = sin(yaw); s_cam[3] = -cos(yaw);
        }
        if (camera_out)
            for (int k = 0; k < 4; k++) camera_out[k] = s_cam[k];
    }
    if (a < 0 || !cars) return;
    const int env = a / A;
    for (int k = threadIdx.x; k < A; k += blockDim.x) {
        const size_t b = (size_t)env * A + k;
        double v[8];
        get_vertices(state[b], state[NA + b], state[4 * NA + b], length, width, v);
        double *c = s_car + F110_RENDER_CAR * k;
        double lx = v[0], hx = v[0], ly = v[1], hy = v[1];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            c[2 * i] = v[2 * i]; c[2 * i + 1] = v[2 * i + 1];
            lx = fmin(lx, v[2 * i]); hx = fmax(hx, v[2 * i]);
            ly = fmin(ly, v[2 * i + 1]); hy = fmax(hy, v[2 * i + 1]);
        }
        const double m = 1e-6 * ((hx - lx) + (hy - ly));
        c[8] = lx - m; c[9] = hx + m; c[10] = ly - m; c[11] = hy + m;
    }
}

// Gather pass: blockIdx.y walks the frames, a thread owns 4 consecutive pixels of a row and stores them as one 32-bit word (labels)
// or three (RGB).  The block puts the frame's camera and the vertices and widened boxes of the viewer's env's A cars in shared
// memory (A * 96 B dynamic).
template <bool FAST>
__global__ void __launch_bounds__(F110_RENDER_THREADS) k_render_frame(RenderArgs r, double *__restrict__ camera_out) {
    extern __shared__ double s_car[];
    __shared__ double s_cam[4];
    const int A = r.num_agents;
    const unsigned gpr = (unsigned)r.W >> 2;                 // 4-pixel groups per row
    const unsigned groups = gpr * (unsigned)r.H;
    const unsigned g = blockIdx.x * blockDim.x + threadIdx.x;
    const size_t frame_bytes = (size_t)r.W * (size_t)r.H * (size_t)r.channels;
    for (int f = blockIdx.y; f < r.num_frames; f += gridDim.y) {
        const int a = render_viewer(r, f);
        render_prepare(r.state, r.num_envs, A, a, r.camera, r.center_x, r.center_y, true, r.length, r.width, s_cam, s_car,
                       (camera_out && blockIdx.x == 0) ? camera_out + 4 * (size_t)f : nullptr);
        __syncthreads();
        if (g < groups) {
            const unsigned row = g / gpr, c0 = (g - row * gpr) * 4;
            uint32_t lab[4] = {0, 0, 0, 0};
            if (a >= 0) {
                const double cx = s_cam[0], cy = s_cam[1], cr = s_cam[2], sr = s_cam[3];
                const int env = a / A, me = a - env * A;
                const double *dt = r.dt;
                if (r.env_layer) dt += (size_t)r.env_layer[env] * r.layer_stride;
                const double v = (0.5 * r.H - (double)row - 0.5) * r.mpp;
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const double u = ((double)(c0 + j) + 0.5 - 0.5 * r.W) * r.mpp;
                    const double x = cx + (u * cr - v * sr);
                    const double y = cy + (u * sr + v * cr);
                    uint32_t l = 0;
                    if (render_in_car(s_car + F110_RENDER_CAR * me, x, y)) {
                        l = 2;
                    } else {
                        for (int k = 0; k < A; k++)
                            if (k != me && render_in_car(s_car + F110_RENDER_CAR * k, x, y)) { l = 3; break; }
                        if (l == 0 && render_wall<FAST>(r, dt, x, y)) l = 1;
                    }
                    lab[j] = l;
                }
            }
            const size_t o = (size_t)f * frame_bytes + ((size_t)row * (size_t)r.W + c0) * (size_t)r.channels;
            if (r.channels == 1) {
                *reinterpret_cast<uint32_t *>(r.out + o) = lab[0] | (lab[1] << 8) | (lab[2] << 16) | (lab[3] << 24);
            } else {
                uint32_t w[3] = {0, 0, 0};
#pragma unroll
                for (int j = 0; j < 4; j++)
#pragma unroll
                    for (int k = 0; k < 3; k++) {
                        const int byte = 3 * j + k;
                        w[byte >> 2] |= (uint32_t)r.palette[lab[j]][k] << (8 * (byte & 3));
                    }
                uint32_t *p = reinterpret_cast<uint32_t *>(r.out + o);
                p[0] = w[0]; p[1] = w[1]; p[2] = w[2];
            }
        }
        __syncthreads();
    }
}

// world point -> its pixel of frame f (dropped when it lands outside the frame), written as `label` / palette[label]
__device__ __forceinline__ void render_plot(const RenderArgs &r, int f, const double cam[4], double px, double py, int label) {
    const double du = px - cam[0], dv = py - cam[1];
    const double u = du * cam[2] + dv * cam[3];
    const double v = -du * cam[3] + dv * cam[2];
    const double fc = floor(u / r.mpp + 0.5 * r.W);
    const double fr = floor(0.5 * r.H - v / r.mpp);
    if (!(fc >= 0.0 && fc < (double)r.W && fr >= 0.0 && fr < (double)r.H)) return;
    const size_t o = ((size_t)f * (size_t)r.H * (size_t)r.W + (size_t)fr * (size_t)r.W + (size_t)fc) * (size_t)r.channels;
    if (r.channels == 1) {
        r.out[o] = (uint8_t)label;
    } else {
        r.out[o] = r.palette[label][0]; r.out[o + 1] = r.palette[label][1]; r.out[o + 2] = r.palette[label][2];
    }
}

// Scan overlay: thread per beam of the frame's viewer (blockIdx.y walks the frames).  Endpoints of ranges < max_range, from the scan
// position along yaw + scan_angles[i], with the pose the scan was taken from (scan_pose / agent_poses of the last tick).
__global__ void __launch_bounds__(F110_RENDER_THREADS) k_render_scan(RenderArgs r, const float *__restrict__ scans,
                                                                     const double *__restrict__ scan_pose,
                                                                     const double *__restrict__ agent_poses,
                                                                     const double *__restrict__ scan_angles, int B,
                                                                     double max_range) {
    __shared__ double s_cam[4];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    for (int f = blockIdx.y; f < r.num_frames; f += gridDim.y) {
        const int a = render_viewer(r, f);
        if (threadIdx.x == 0)
            render_prepare(r.state, r.num_envs, r.num_agents, a, r.camera, r.center_x, r.center_y, false, 0.0, 0.0, s_cam,
                           nullptr, nullptr);
        __syncthreads();
        if (a >= 0 && i < B) {
            const double rng = (double)scans[(size_t)a * B + i];
            if (rng < max_range) {
                const double th = agent_poses[5 * (size_t)a + 2] + scan_angles[i];
                const double px = scan_pose[4 * (size_t)a] + rng * cos(th);
                const double py = scan_pose[4 * (size_t)a + 1] + rng * sin(th);
                render_plot(r, f, s_cam, px, py, 4);
            }
        }
        __syncthreads();
    }
}

// Waypoint overlay: thread per (frame, waypoint row).  table_start == NULL: every frame draws all rows; else row w belongs to table
// t when table_start[t] <= w < table_start[t + 1] and a frame draws the table env_table[env] of its viewer's env.
__global__ void __launch_bounds__(F110_RENDER_THREADS) k_render_waypoints(RenderArgs r, const double *__restrict__ wx,
                                                                          const double *__restrict__ wy, int num_waypoints,
                                                                          const int32_t *__restrict__ table_start,
                                                                          int num_tables,
                                                                          const int32_t *__restrict__ env_table) {
    __shared__ double s_cam[4];
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    for (int f = blockIdx.y; f < r.num_frames; f += gridDim.y) {
        const int a = render_viewer(r, f);
        if (threadIdx.x == 0)
            render_prepare(r.state, r.num_envs, r.num_agents, a, r.camera, r.center_x, r.center_y, false, 0.0, 0.0, s_cam,
                           nullptr, nullptr);
        __syncthreads();
        if (a >= 0 && w < num_waypoints) {
            bool mine = true;
            if (table_start) {
                const int t = env_table[a / r.num_agents];
                mine = t >= 0 && t < num_tables && w >= table_start[t] && w < table_start[t + 1];
            }
            if (mine) render_plot(r, f, s_cam, wx[w], wy[w], 5);
        }
        __syncthreads();
    }
}

}  // namespace f110
