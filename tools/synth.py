"""Deterministic synthetic LiDAR workload (SURVEY.md 8d): an analytic street scene ray-cast exactly, in the style
of the reference's own generator (mapping/internal/3d/local_trajectory_builder_3d_test.cc:117-250) scaled to street
size. numpy only; used by tests/ and bench.py to produce RangeMeasurement rows of the named shapes.

Scene (seed 42): ground plane z = -1.8 m, facade planes y = +-12 m, 64 axis-aligned boxes (2-10 m), 100 spheres
r = 0.5 m. Range noise N(0, 0.02 m) (seed 43). Sensors: 16-beam (+-15 deg, 1800 az = 28 800 pts), 64-beam
(+2 .. -24.8 deg, 2048 az = 131 072 pts), 128-beam (+-22.5 deg, 2048 az = 262 144 pts); 10 Hz, per-point time in
[-0.1, 0] with the last point at 0 (timed_point_cloud_data.h contract, LTB:384).
Trajectory: 10 m/s along +x with a 0.2 rad/s-amplitude yaw sinusoid; the sensor moves during the sweep.
"""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
RAYCAST_LIB = os.path.join(_HERE, "libraycast.so")
_RAYCAST = None


def build_raycast(path=RAYCAST_LIB):
    """Compiles raycast.c into `path` (__graft_entry__.build() makes tools/libraycast.so)."""
    subprocess.check_call(["gcc", "-O2", "-fopenmp", "-shared", "-fPIC", "-o", path, os.path.join(_HERE, "raycast.c"), "-lm"])


def _raycast_lib():
    """tools/libraycast.so (C, OpenMP): ~40x faster than the numpy path, optional. In a tree that was not built it is compiled
    into a temporary directory, never into the tree (which may be read-only)."""
    global _RAYCAST
    if _RAYCAST is None:
        try:
            if os.path.exists(RAYCAST_LIB):
                L = ctypes.CDLL(RAYCAST_LIB)
            else:
                with tempfile.TemporaryDirectory() as d:
                    path = os.path.join(d, "libraycast.so")
                    build_raycast(path)
                    L = ctypes.CDLL(path)   # stays mapped after the directory is removed
            dp = np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS")
            L.synth_raycast.argtypes = [ctypes.c_int64, dp, dp, ctypes.c_double, ctypes.c_double, ctypes.c_int, dp, dp,
                                        ctypes.c_int, dp, ctypes.c_double, ctypes.c_double, dp]
            _RAYCAST = L
        except Exception:  # no compiler: fall back to numpy (data generation only, never the measured path)
            _RAYCAST = False
    return _RAYCAST

SENSORS = {
    16: dict(beams=16, az=1800, elev=(-15.0, 15.0)),
    64: dict(beams=64, az=2048, elev=(-24.8, 2.0)),
    128: dict(beams=128, az=2048, elev=(-22.5, 22.5)),
}
RANGE_DTYPE = np.dtype([("x", np.float32), ("y", np.float32), ("z", np.float32), ("t", np.float32),
                        ("origin_index", np.uint64), ("_pad", np.uint64)])


class Scene:
    def __init__(self, seed=42):
        rng = np.random.RandomState(seed)
        n_box, n_sph = 64, 100
        centers = np.stack([rng.uniform(-20, 220, n_box), rng.uniform(4.0, 11.0, n_box) * rng.choice([-1, 1], n_box),
                            np.zeros(n_box)], 1)
        half = rng.uniform(1.0, 5.0, (n_box, 3))
        half[:, 1] = np.minimum(half[:, 1], 2.0)     # keep the driving corridor |y| < 2 free
        centers[:, 2] = -1.8 + half[:, 2]
        self.box_lo, self.box_hi = centers - half, centers + half
        self.sph_c = np.stack([rng.uniform(-20, 220, n_sph), rng.uniform(3.0, 11.5, n_sph) * rng.choice([-1, 1], n_sph),
                               rng.uniform(-1.3, 4.0, n_sph)], 1)
        self.sph_r = 0.5
        self.ground_z, self.facade_y = -1.8, 12.0

    def raycast(self, origins, dirs, max_range=150.0):
        """origins, dirs: (n, 3) float64, dirs unit. Returns ranges (inf = no hit)."""
        n = len(dirs)
        L = _raycast_lib()
        if L:
            out = np.zeros(n)
            L.synth_raycast(n, np.ascontiguousarray(origins, np.float64), np.ascontiguousarray(dirs, np.float64),
                            self.ground_z, self.facade_y, len(self.box_lo), np.ascontiguousarray(self.box_lo),
                            np.ascontiguousarray(self.box_hi), len(self.sph_c), np.ascontiguousarray(self.sph_c),
                            self.sph_r, max_range, out)
            return out
        best = np.full(n, np.inf)
        with np.errstate(divide="ignore", invalid="ignore"):
            t = (self.ground_z - origins[:, 2]) / dirs[:, 2]
            best = np.where((t > 0) & (t < best), t, best)
            for y in (self.facade_y, -self.facade_y):
                t = (y - origins[:, 1]) / dirs[:, 1]
                best = np.where((t > 0) & (t < best), t, best)
            inv = 1.0 / dirs
            for lo, hi in zip(self.box_lo, self.box_hi):
                t1, t2 = (lo - origins) * inv, (hi - origins) * inv
                tn, tf = np.minimum(t1, t2).max(1), np.maximum(t1, t2).min(1)
                hit = (tn <= tf) & (tn > 0) & (tn < best)
                best = np.where(hit, tn, best)
            for c in self.sph_c:
                oc = origins - c
                b = (oc * dirs).sum(1)
                disc = b * b - ((oc * oc).sum(1) - self.sph_r ** 2)
                t = -b - np.sqrt(np.where(disc > 0, disc, np.nan))
                hit = (disc > 0) & (t > 0) & (t < best)
                best = np.where(hit, t, best)
        best[best > max_range] = np.inf
        return best


def trajectory_pose(t):
    """(position (.., 3), yaw) of the tracking frame at time t (seconds, array ok)."""
    t = np.asarray(t, np.float64)
    yaw = 0.2 * np.sin(0.5 * t) * 0.8
    pos = np.stack([10.0 * t, 0.6 * np.sin(0.3 * t), np.zeros_like(t)], -1)
    return pos, yaw


def pose7(t):
    pos, yaw = trajectory_pose(t)
    return np.array([pos[0], pos[1], pos[2], np.cos(yaw / 2), 0.0, 0.0, np.sin(yaw / 2)])


def make_scan(scene, beams, scan_end_time, scan_period=0.1, noise_seed=43, noise_sigma=0.02):
    """One sweep ending at scan_end_time. Returns RangeMeasurement rows (points in the tracking frame AT THE
    TIME OF EACH POINT, as a real spinning LiDAR delivers them) with per-point time in [-period, 0]."""
    s = SENSORS[beams]
    az = np.linspace(0.0, 2 * np.pi, s["az"], endpoint=False)
    el = np.deg2rad(np.linspace(s["elev"][0], s["elev"][1], s["beams"]))
    A, E = np.meshgrid(az, el, indexing="ij")      # azimuth-major: time increases with azimuth
    A, E = A.ravel(), E.ravel()
    n = len(A)
    tp = (np.arange(n) // s["beams"]).astype(np.float64)
    t_rel = -scan_period * (1.0 - (tp + 1) / s["az"])     # last column -> 0
    dirs_s = np.stack([np.cos(E) * np.cos(A), np.cos(E) * np.sin(A), np.sin(E)], 1)
    pos, yaw = trajectory_pose(scan_end_time + t_rel)
    c, sn = np.cos(yaw), np.sin(yaw)
    dirs_w = np.stack([c * dirs_s[:, 0] - sn * dirs_s[:, 1], sn * dirs_s[:, 0] + c * dirs_s[:, 1], dirs_s[:, 2]], 1)
    r = scene.raycast(pos, dirs_w)
    rng = np.random.RandomState(noise_seed + int(round(scan_end_time * 1000)) % 100000)
    r = r + rng.normal(0.0, noise_sigma, n)
    ok = np.isfinite(r) & (r > 0.3)
    pts = dirs_s[ok] * r[ok, None]
    rows = np.zeros(int(ok.sum()), RANGE_DTYPE)
    rows["x"], rows["y"], rows["z"] = pts[:, 0], pts[:, 1], pts[:, 2]
    rows["t"] = t_rel[ok]
    rows["t"][-1] = 0.0
    return rows


def perturb_pose(p7, rng, dt=0.1, dr_deg=1.0):
    """Initial-pose perturbation for matcher benches: uniform +-dt m, +-dr_deg degrees (seed 45 in the callers)."""
    out = np.array(p7, np.float64)
    out[:3] += rng.uniform(-dt, dt, 3)
    aa = np.deg2rad(rng.uniform(-dr_deg, dr_deg, 3))
    ang = np.linalg.norm(aa)
    dq = np.array([1.0, 0, 0, 0]) if ang == 0 else np.concatenate([[np.cos(ang / 2)], np.sin(ang / 2) * aa / ang])
    w, x, y, z = out[3:]
    a = dq
    out[3:] = [a[0] * w - a[1] * x - a[2] * y - a[3] * z, a[0] * x + a[1] * w + a[2] * z - a[3] * y,
               a[0] * y - a[1] * z + a[2] * w + a[3] * x, a[0] * z + a[1] * y - a[2] * x + a[3] * w]
    out[3:] /= np.linalg.norm(out[3:])
    return out
