"""Seeded synthetic scenes for parity tests and bench.py (SURVEY.md §8d): a piecewise-planar "city grid" world,
spinning / rosette LiDAR ray casting, a voxel-resolution map pre-fill and state helpers.  Host-side numpy data
generation only — no part of the measured path.

The reference ships no data (SURVEY.md §4), so every input is generated here from a seed.
"""
import numpy as np

G_LEN = 9.809  # |grav| of MTK::S2<double, 98090, 10000, 1> (include/use-ikfom.hpp:8)


# ----------------------------------------------------------------------------------------------- world
class World:
    """Axis-aligned rectangles: (axis, coord, (lo_u, hi_u), (lo_v, hi_v)) with (u,v) = the other two axes in order."""

    def __init__(self):
        self.axis, self.coord, self.lo, self.hi = [], [], [], []

    def add(self, axis, coord, lo_uv, hi_uv):
        self.axis.append(axis)
        self.coord.append(coord)
        self.lo.append(lo_uv)
        self.hi.append(hi_uv)

    def finalize(self):
        self.axis = np.asarray(self.axis, np.int64)
        self.coord = np.asarray(self.coord, np.float64)
        self.lo = np.asarray(self.lo, np.float64).reshape(-1, 2)
        self.hi = np.asarray(self.hi, np.float64).reshape(-1, 2)
        return self

    def shifted(self, d):
        """The same world translated by d = (dx, dy, dz) (call after finalize)."""
        d = np.asarray(d, np.float64)
        w = World()
        w.axis = self.axis.copy()
        w.coord = self.coord + d[self.axis]
        uv = np.array([_OTHER[int(a)] for a in self.axis], np.int64).reshape(-1, 2)
        w.lo = self.lo + d[uv]
        w.hi = self.hi + d[uv]
        return w

    def add_box(self, lo, hi):
        """Four walls and a roof of a building lo=(x0,y0,z0), hi=(x1,y1,z1)."""
        (x0, y0, z0), (x1, y1, z1) = lo, hi
        self.add(0, x0, (y0, z0), (y1, z1))
        self.add(0, x1, (y0, z0), (y1, z1))
        self.add(1, y0, (x0, z0), (x1, z1))
        self.add(1, y1, (x0, z0), (x1, z1))
        self.add(2, z1, (x0, y0), (x1, y1))


def city_world(half_extent=300.0, pitch=60.0, street=16.0, seed=0, clutter=True):
    """Ground plane z=0 plus a grid of buildings (pitch x pitch cells, `street` wide streets) with seeded heights,
    and small clutter boxes (parked cars / kiosks) along the streets."""
    rng = np.random.default_rng(seed)
    w = World()
    e = half_extent
    w.add(2, 0.0, (-e, -e), (e, e))
    n = int(np.ceil(e / pitch))
    for i in range(-n, n):
        for j in range(-n, n):
            x0 = i * pitch + street / 2
            y0 = j * pitch + street / 2
            x1 = (i + 1) * pitch - street / 2
            y1 = (j + 1) * pitch - street / 2
            h = rng.uniform(6.0, 18.0)
            # jitter the footprint a little so facades are not coplanar across blocks
            jx0, jy0, jx1, jy1 = rng.uniform(0.0, 3.0, 4)
            w.add_box((x0 + jx0, y0 + jy0, 0.0), (x1 - jx1, y1 - jy1, h))
            if clutter:
                for _ in range(3):
                    cx = rng.uniform(i * pitch - street / 2 + 1.0, i * pitch + street / 2 - 3.0)
                    cy = rng.uniform(j * pitch + street / 2, (j + 1) * pitch - street / 2 - 5.0)
                    w.add_box((cx, cy, 0.0), (cx + rng.uniform(1.5, 2.2), cy + rng.uniform(3.5, 5.0), rng.uniform(1.2, 2.0)))
    return w.finalize()


_OTHER = {0: (1, 2), 1: (0, 2), 2: (0, 1)}


def raycast(world, origin, dirs_world, max_range=100.0, min_range=1.0):
    """Nearest hit distance per ray (inf if none within [min_range, max_range])."""
    o = np.asarray(origin, np.float64)
    d = np.asarray(dirs_world, np.float64)
    n = len(d)
    best = np.full(n, np.inf)
    # cull rectangles farther than max_range from the origin
    for ax in (0, 1, 2):
        u, v = _OTHER[ax]
        idx = np.nonzero(world.axis == ax)[0]
        if len(idx) == 0:
            continue
        c = world.coord[idx]
        lo, hi = world.lo[idx], world.hi[idx]
        du = np.maximum(np.maximum(lo[:, 0] - o[u], o[u] - hi[:, 0]), 0)
        dv = np.maximum(np.maximum(lo[:, 1] - o[v], o[v] - hi[:, 1]), 0)
        near = np.sqrt((c - o[ax]) ** 2 + du ** 2 + dv ** 2) <= max_range
        idx = idx[near]
        if len(idx) == 0:
            continue
        c, lo, hi = world.coord[idx], world.lo[idx], world.hi[idx]
        da = d[:, ax]
        with np.errstate(divide="ignore", invalid="ignore"):
            for k in range(len(idx)):
                t = (c[k] - o[ax]) / da
                ok = (t > min_range) & (t < best)
                if not ok.any():
                    continue
                hu = o[u] + t * d[:, u]
                hv = o[v] + t * d[:, v]
                ok &= (hu >= lo[k, 0]) & (hu <= hi[k, 0]) & (hv >= lo[k, 1]) & (hv <= hi[k, 1])
                best = np.where(ok, t, best)
    best[best > max_range] = np.inf
    return best


# ----------------------------------------------------------------------------------------------- sensors
def lidar_dirs(model, rng=None):
    """Unit ray directions in the LiDAR frame."""
    if model == "vlp16":      # 16 rings +-15 deg, 1800 azimuth steps -> 28 800 rays
        el = np.deg2rad(np.linspace(-15, 15, 16))
        az = np.deg2rad(np.arange(1800) * 0.2)
    elif model == "hdl64":    # 64 rings +2 .. -24.8 deg, 1875 azimuth steps -> 120 000 rays
        el = np.deg2rad(np.linspace(2.0, -24.8, 64))
        az = np.deg2rad(np.arange(1875) * (360.0 / 1875))
    elif model == "os64":     # Ouster-64: 64 x 1024, +-16.6 deg
        el = np.deg2rad(np.linspace(16.6, -16.6, 64))
        az = np.deg2rad(np.arange(1024) * (360.0 / 1024))
    elif model == "hap":      # Livox HAP: 120 x 25 deg FoV, non-repetitive -> 240 000 random rays
        rng = rng or np.random.default_rng(0)
        a = np.deg2rad(rng.uniform(-60, 60, 240000))
        e = np.deg2rad(rng.uniform(-12.5, 12.5, 240000))
        return np.stack([np.cos(e) * np.cos(a), np.cos(e) * np.sin(a), np.sin(e)], 1)
    else:
        raise ValueError(model)
    E, A = np.meshgrid(el, az, indexing="ij")
    return np.stack([(np.cos(E) * np.cos(A)).ravel(), (np.cos(E) * np.sin(A)).ravel(), np.sin(E).ravel()], 1)


def quat_mul(a, b):
    ax, ay, az, aw = a
    bx, by, bz, bw = b
    return np.array([aw * bx + ax * bw + ay * bz - az * by, aw * by + ay * bw + az * bx - ax * bz,
                     aw * bz + az * bw + ax * by - ay * bx, aw * bw - ax * bx - ay * by - az * bz])


def quat_from_rotvec(v):
    v = np.asarray(v, np.float64)
    th = np.linalg.norm(v)
    if th < 1e-12:
        return np.array([v[0] / 2, v[1] / 2, v[2] / 2, 1.0])
    s = np.sin(th / 2) / th
    return np.array([v[0] * s, v[1] * s, v[2] * s, np.cos(th / 2)])


def quat_to_mat(q):
    x, y, z, w = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


def make_state(pos=(0, 0, 0), rot=(0, 0, 0, 1), offR=(0, 0, 0, 1), offT=(0.04165, 0.02326, -0.0284), vel=(0, 0, 0),
               bg=(0, 0, 0), ba=(0, 0, 0), grav=(0, 0, -G_LEN)):
    """state26 layout of include/fastlio_b200.h (state_ikfom, use-ikfom.hpp:21-30)."""
    return np.concatenate([pos, rot, offR, offT, vel, bg, ba, grav]).astype(np.float64)


def perturb_state(state, rng, sig_pos=0.05, sig_rot_deg=0.5):
    s = state.copy()
    s[0:3] += rng.normal(0, sig_pos, 3)
    dq = quat_from_rotvec(rng.normal(0, np.deg2rad(sig_rot_deg), 3))
    q = quat_mul(s[3:7], dq)
    s[3:7] = q / np.linalg.norm(q)
    return s


def default_cov():
    """Prior covariance of a propagated state (diagonal; orders of magnitude of IMU_Processing.hpp:224-231 grown by
    one propagation step)."""
    d = np.zeros(23)
    d[0:3] = 2.5e-3
    d[3:6] = 8e-5
    d[6:9] = 1e-5
    d[9:12] = 1e-5
    d[12:15] = 1e-2
    d[15:18] = 1e-4
    d[18:21] = 1e-3
    d[21:23] = 1e-5
    return np.diag(d)


def scan_from_pose(world, state_true, dirs_lidar, rng, max_range=100.0, min_range=2.0, noise=0.01):
    """Ray-cast one scan from the TRUE state; returns float32 points in the LiDAR (body) frame, range noise sigma."""
    R = quat_to_mat(state_true[3:7])
    Rli = quat_to_mat(state_true[7:11])
    o = state_true[0:3] + R @ state_true[11:14]
    dw = dirs_lidar @ (R @ Rli).T
    t = raycast(world, o, dw, max_range, min_range)
    ok = np.isfinite(t)
    t = t[ok] + rng.normal(0, noise, ok.sum())
    return (dirs_lidar[ok] * t[:, None]).astype(np.float32)


def body_to_world_np(state, body):
    R = quat_to_mat(state[3:7])
    Rli = quat_to_mat(state[7:11])
    return ((body.astype(np.float64) @ Rli.T + state[11:14]) @ R.T + state[0:3]).astype(np.float32)


def voxel_downsample(pts, leaf):
    """pcl::VoxelGrid stand-in (centroid per voxel) — the step BEFORE the path (laserMapping.cpp:2322-2323)."""
    if len(pts) == 0:
        return pts
    k = np.floor(pts / leaf).astype(np.int64)
    key = (k[:, 0] * 73856093) ^ (k[:, 1] * 19349663) ^ (k[:, 2] * 83492791)
    order = np.argsort(key, kind="stable")
    ks = key[order]
    start = np.r_[0, np.nonzero(ks[1:] != ks[:-1])[0] + 1]
    cnt = np.diff(np.r_[start, len(ks)])
    sums = np.add.reduceat(pts[order].astype(np.float64), start, axis=0)
    return (sums / cnt[:, None]).astype(np.float32)


def sample_surface_map(world, center, half, ds, rng, noise=0.01, zmax=25.0):
    """Map pre-fill: about one jittered point per ds x ds cell on every surface inside the box |p - center| <= half
    (half: scalar or per-axis)
    (what map_incremental converges to: one point per filter_size_map_min voxel, SURVEY.md §3.3)."""
    out = []
    c = np.asarray(center, np.float64)
    hv = np.broadcast_to(np.asarray(half, np.float64), (3,)) if np.ndim(half) else np.full(3, float(half))
    for k in range(len(world.axis)):
        ax = int(world.axis[k])
        u, v = _OTHER[ax]
        if abs(world.coord[k] - c[ax]) > hv[ax]:
            continue
        lo = np.maximum(world.lo[k], [c[u] - hv[u], c[v] - hv[v]])
        hi = np.minimum(world.hi[k], [c[u] + hv[u], c[v] + hv[v]])
        if v == 2:
            hi[1] = min(hi[1], zmax)
        if ax == 2 and world.coord[k] > zmax:
            continue
        if hi[0] <= lo[0] or hi[1] <= lo[1]:
            continue
        nu = max(int((hi[0] - lo[0]) / ds), 1)
        nv = max(int((hi[1] - lo[1]) / ds), 1)
        U, V = np.meshgrid(np.arange(nu), np.arange(nv), indexing="ij")
        pu = lo[0] + (U.ravel() + rng.uniform(0.05, 0.95, nu * nv)) * ds
        pv = lo[1] + (V.ravel() + rng.uniform(0.05, 0.95, nu * nv)) * ds
        p = np.empty((nu * nv, 3))
        p[:, ax] = world.coord[k] + rng.normal(0, noise, nu * nv)
        p[:, u] = pu
        p[:, v] = pv
        out.append(p)
    if not out:
        return np.zeros((0, 3), np.float32)
    return np.concatenate(out).astype(np.float32)


def trajectory_state(k, speed=10.0, dt=0.1, z=1.8, yaw_amp_deg=4.0, start=(0.0, 0.0)):
    """True state of scan k: drive along +x through the street at y = start[1] with a gentle yaw oscillation."""
    x = start[0] + speed * dt * k
    yaw = np.deg2rad(yaw_amp_deg) * np.sin(0.05 * k)
    q = quat_from_rotvec([0.0, 0.0, yaw])
    y = start[1] + 1.5 * np.sin(0.02 * k)
    return make_state(pos=(x, y, z), rot=q, vel=(speed, 0, 0))


# ------------------------------------------------------------------------------------------------ front-end inputs
def imu_pose_sequence(state0, rng, n_imu=21, scan_time=0.1, first_offset=0.002):
    """A plausible IMUpose vector (IMU_Processing.hpp:260-322) for one scan: n_imu+1 Pose6D records of 22 doubles
    (offset_time, acc[3], gyr[3], vel[3], pos[3], rot[9] row-major); record 0 is the previous posterior at offset 0.
    Returns (poses[n_imu+1,22], state26_end) where state26_end is the propagated state at the last record."""
    st = np.array(state0, np.float64).copy()
    R = quat_to_mat(st[3:7])
    vel = np.array([10.0, 0.3, 0.0]) + rng.normal(0, 0.1, 3)
    pos = st[0:3].copy()
    gyr = np.array([0.02, -0.03, 0.25]) + rng.normal(0, 0.02, 3)
    acc = np.array([0.4, -0.2, 0.1]) + rng.normal(0, 0.05, 3)
    poses = [np.concatenate([[0.0], acc, gyr, vel, pos, R.reshape(-1)])]
    t_prev = 0.0
    for k in range(n_imu):
        t = first_offset + k * (scan_time / max(n_imu - 1, 1))
        dt = t - t_prev
        g = gyr + rng.normal(0, 0.01, 3)
        a = acc + rng.normal(0, 0.05, 3)
        R = R @ quat_to_mat(quat_from_rotvec(g * dt))
        pos = pos + vel * dt + 0.5 * a * dt * dt
        vel = vel + a * dt
        poses.append(np.concatenate([[t], a, g, vel, pos, R.reshape(-1)]))
        t_prev = t
    end = st.copy()
    end[0:3] = pos
    end[14:17] = vel
    # rotation matrix -> quaternion (x,y,z,w)
    w = np.sqrt(max(0.0, 1.0 + R[0, 0] + R[1, 1] + R[2, 2])) / 2.0
    end[3:7] = [(R[2, 1] - R[1, 2]) / (4 * w), (R[0, 2] - R[2, 0]) / (4 * w), (R[1, 0] - R[0, 1]) / (4 * w), w]
    return np.array(poses, np.float64), end


def raw_scan_with_times(body_xyz, rng, scan_time_ms=100.0, shuffle=True):
    """Attach intensity and per-point time offsets (curvature, ms — preprocess.cpp) to a scan; the returns arrive in
    azimuth order with a few exact zeros and exact duplicates, as real drivers produce."""
    n = len(body_xyz)
    az = np.arctan2(body_xyz[:, 1], body_xyz[:, 0])
    cur = ((az + np.pi) / (2 * np.pi) * scan_time_ms).astype(np.float32)
    cur[rng.integers(0, n, max(1, n // 500))] = 0.0
    cur = np.round(cur * 8.0) / 8.0   # quantised stamps -> many exact ties
    inten = rng.uniform(0, 255, n).astype(np.float32)
    order = rng.permutation(n) if shuffle else np.arange(n)
    return body_xyz[order].astype(np.float32), inten[order], cur[order].astype(np.float32)


# ----------------------------------------------------------------------------------------------- driver records
def sensor_scan(world, model, rng, columns=None, origin=(0.0, 0.0, 1.8), max_range=100.0, min_range=1.0):
    """Returns of one sweep in the order the driver sends them: for spinning sensors column by column (all rings of
    one azimuth, then the next; azimuth decreasing, i.e. clockwise as Velodyne and Ouster spin), for Livox in firing
    order.  `columns` keeps that many azimuth columns spread over the full turn (spinning) or the first that many
    returns (Livox).  Returns xyz (float32), ring (int) and the azimuth column
    (spinning) or firing index (Livox) of every return; rays without a hit are dropped."""
    d = lidar_dirs(model, rng)
    if model == "hap":
        if columns is not None:
            d = d[:columns]
        ring = np.arange(len(d)) % 6
        col = np.arange(len(d))
    else:
        n_rings = {"vlp16": 16, "hdl64": 64, "os64": 64}[model]
        d = d.reshape(n_rings, -1, 3)
        d = d[:, ::-1]
        if columns is not None:
            d = d[:, ::max(1, d.shape[1] // columns)][:, :columns]
        n_cols = d.shape[1]
        d = d.transpose(1, 0, 2).reshape(-1, 3)            # column-major: rings interleaved
        ring = np.tile(np.arange(n_rings), n_cols)
        col = np.repeat(np.arange(n_cols), n_rings)
    r = raycast(world, origin, d, max_range=max_range, min_range=min_range)
    ok = np.isfinite(r)
    xyz = (d[ok] * r[ok, None]).astype(np.float32)
    return xyz, ring[ok], col[ok]


def velodyne_records(xyz, ring, time_s, rng):
    from .capi import VELODYNE_RECORD
    rec = np.zeros(len(xyz), VELODYNE_RECORD)
    rec["x"], rec["y"], rec["z"] = xyz[:, 0], xyz[:, 1], xyz[:, 2]
    rec["intensity"] = rng.integers(0, 256, len(xyz)).astype(np.float32)
    rec["time"] = time_s
    rec["ring"] = ring
    return rec


def ouster_records(xyz, ring, t_int, rng):
    from .capi import OUSTER_RECORD
    rec = np.zeros(len(xyz), OUSTER_RECORD)
    rec["x"], rec["y"], rec["z"] = xyz[:, 0], xyz[:, 1], xyz[:, 2]
    rec["intensity"] = rng.uniform(0, 3000, len(xyz)).astype(np.float32)
    rec["t"] = t_int
    rec["ring"] = ring
    rec["reflectivity"] = rng.integers(0, 65536, len(xyz))
    rec["range"] = (np.linalg.norm(xyz, axis=1) * 1000).astype(np.uint32)
    return rec


def livox_records(xyz, line, offset_ns, rng, tag_mix=True):
    """CustomMsg points; with tag_mix, about 10 % carry a second/third-return or noise tag."""
    from .capi import LIVOX_RECORD
    rec = np.zeros(len(xyz), LIVOX_RECORD)
    rec["x"], rec["y"], rec["z"] = xyz[:, 0], xyz[:, 1], xyz[:, 2]
    rec["reflectivity"] = rng.integers(0, 256, len(xyz))
    rec["offset_time"] = offset_ns
    rec["line"] = line
    if tag_mix:
        rec["tag"] = rng.choice(np.array([0x00, 0x10, 0x20, 0x30, 0x01, 0x12, 0x24], np.uint8), len(xyz),
                                p=[0.6, 0.2, 0.05, 0.05, 0.04, 0.04, 0.02])
    return rec
