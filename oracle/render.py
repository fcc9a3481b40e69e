"""numpy restatement of the headless renderer (f1tenth_gym_b200/csrc/render.cuh, C ABI f110_render).

TEST AND MEASUREMENT INFRASTRUCTURE ONLY, like the C oracle: tests/ and tools/render_bench.py compare the device frames
against it.  Every expression keeps the kernel's operation order in fp64 (numpy elementwise arithmetic contracts nothing into
an FMA, and the library is built with -fmad=false), so labels match bit for bit when the inputs do: the tests feed it the
vertices of f110_get_vertices and the cameras of camera_out rather than recomputing sin / cos here.

Labels: 0 free / off the map, 1 wall, 2 the viewer's car, 3 other cars of its env, 4 scan endpoints, 5 waypoints.
"""
import numpy as np

FREE, WALL, VIEWER, OTHER_CAR, SCAN, WAYPOINT = range(6)


def pixel_centres(cam, width, height, mpp):
    """World (x, y), each [height][width], of the pixel centres of a frame with camera (cx, cy, cr, sr)."""
    cx, cy, cr, sr = (float(v) for v in cam)
    u = ((np.arange(width, dtype=np.float64) + 0.5) - 0.5 * width) * mpp
    v = ((0.5 * height - np.arange(height, dtype=np.float64)) - 0.5) * mpp
    U, V = u[None, :], v[:, None]
    return cx + (U * cr - V * sr), cy + (U * sr + V * cr)


def walls(dt, resolution, orig_x, orig_y, orig_c, orig_s, x, y):
    """Literal xy_2_rc (reference laser_models.py:55-86) of every point; True where the cell's dt == 0.  Off the map (and an
    index that rounds up to the table's size, or NaN) is free."""
    mh, mw = dt.shape
    tx, ty = x - orig_x, y - orig_y
    xr = tx * orig_c + ty * orig_s
    yr = -tx * orig_s + ty * orig_c
    with np.errstate(invalid='ignore'):
        inb = (xr >= 0) & (xr < mw * resolution) & (yr >= 0) & (yr < mh * resolution)
    c = np.where(inb, xr / resolution, 0.0).astype(np.int64)
    r = np.where(inb, yr / resolution, 0.0).astype(np.int64)
    inb &= (c < mw) & (r < mh)
    return inb & (dt[np.where(inb, r, 0), np.where(inb, c, 0)] == 0.0)


def inside_car(v, x, y):
    """v [8] = (rl, rr, fr, fl) vertices: all four edge functions (b - a) x (p - a) >= 0."""
    ok = np.ones(np.shape(x), dtype=bool)
    for i in range(4):
        j = (i + 1) % 4
        ax, ay, bx, by = v[2 * i], v[2 * i + 1], v[2 * j], v[2 * j + 1]
        with np.errstate(invalid='ignore'):
            ok &= ((bx - ax) * (y - ay) - (by - ay) * (x - ax)) >= 0.0
    return ok


def base_labels(cam, width, height, mpp, verts, me, dt, resolution, orig_x, orig_y, orig_c, orig_s):
    """Labels 0-3 of one frame.  verts [A][8]: the cars of the viewer's env; me: the viewer's agent slot in it."""
    x, y = pixel_centres(cam, width, height, mpp)
    lab = np.where(walls(dt, resolution, orig_x, orig_y, orig_c, orig_s, x, y), WALL, FREE).astype(np.uint8)
    for k in range(len(verts)):
        if k != me:
            lab[inside_car(verts[k], x, y)] = OTHER_CAR
    lab[inside_car(verts[me], x, y)] = VIEWER
    return lab


def point_pixels(cam, width, height, mpp, px, py):
    """World points -> (row, col, inside, fractional row, fractional col): pixel c = floor(u / mpp + 0.5 W),
    r = floor(0.5 H - v / mpp) in camera coordinates (u, v)."""
    cx, cy, cr, sr = (float(v) for v in cam)
    du, dv = np.asarray(px, np.float64) - cx, np.asarray(py, np.float64) - cy
    u = du * cr + dv * sr
    v = -du * sr + dv * cr
    fc = u / mpp + 0.5 * width
    fr = 0.5 * height - v / mpp
    c, r = np.floor(fc), np.floor(fr)
    inside = (c >= 0) & (c < width) & (r >= 0) & (r < height)
    return np.where(inside, r, 0).astype(np.int64), np.where(inside, c, 0).astype(np.int64), inside, fr, fc


def draw_points(lab, cam, mpp, px, py, label):
    r, c, inside, _, _ = point_pixels(cam, lab.shape[1], lab.shape[0], mpp, px, py)
    lab[r[inside], c[inside]] = label
    return lab


def scan_endpoints(scan_x, scan_y, yaw, scan_angles, ranges, max_range):
    """Endpoints of the ranges < max_range: from the scan position along yaw + scan_angles[i]."""
    rng = np.asarray(ranges, dtype=np.float64)
    keep = rng < max_range
    th = yaw + np.asarray(scan_angles, np.float64)[keep]
    return scan_x + rng[keep] * np.cos(th), scan_y + rng[keep] * np.sin(th)


def rgb(lab, palette):
    return np.asarray(palette, dtype=np.uint8)[lab]
