"""Synthetic ETH-CVG-shaped frame pairs (the dataset is not redistributable / not available offline).

Shape follows the reference's inputs: 640x480 8-bit grayscale + uint16 depth with depth_factor 5000
(config_eth_cvg.yaml:13-18, NID_pose_estimation.cpp:91-106), a ground-truth T_wc per frame, and a
gamma/affine illumination change on frame 1. Everything is an analytic function of a seed, so the
same pair can be regenerated on the GPU box without shipping images.

Scene: height field Z = Z0 + relief(X, Y) in the world frame, textured with a seeded sum of
sinusoids tex(X, Y). Both frames are rendered exactly by ray / height-field intersection (Newton).
Poses are column-major 4x4 (Eigen `.data()` layout, which is what the reference hands to CUDA).
"""
from __future__ import annotations

import dataclasses
import numpy as np

FX, FY, CX, CY = 481.20, -480.0, 319.5, 239.5  # config_eth_cvg.yaml:15-18
DEPTH_FACTOR = 1.0 / 5000  # NID_pose_estimation.cpp:73 (1.0/(int)5000)


@dataclasses.dataclass
class Pair:
    im0: np.ndarray        # uint8 [R,C]
    im1: np.ndarray        # uint8 [R,C]
    depth0: np.ndarray     # float64 [R,C] metres (= uint16 * DEPTH_FACTOR)
    depth0_u16: np.ndarray  # uint16 [R,C]
    T_wc0: np.ndarray      # float64 [16] column-major
    T_wc1: np.ndarray      # float64 [16] column-major
    intr: np.ndarray       # float64 [5] fx,fy,cx,cy,depth_factor
    rows: int
    cols: int


def _rot(rx, ry, rz):
    cx, sx = np.cos(rx), np.sin(rx)
    cy, sy = np.cos(ry), np.sin(ry)
    cz, sz = np.cos(rz), np.sin(rz)
    Rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
    Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
    Rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]])
    return Rx @ Ry @ Rz


class _Scene:
    def __init__(self, rng: np.random.Generator):
        # relief: 3 long waves, total amplitude <= 0.45 m around Z0 = 2.6 m
        self.z0 = 2.6
        self.rk = rng.uniform(1.2, 2.4, size=(3, 2)) * rng.choice([-1, 1], size=(3, 2))
        self.ra = rng.uniform(0.08, 0.15, size=3)
        self.rp = rng.uniform(0, 2 * np.pi, size=3)
        # texture: 4 octaves x 10 waves, wavelengths 1.6 m .. 0.09 m (~300 .. 17 px at 2.6 m), 1/f amplitudes
        ks, amps = [], []
        for octave in range(4):
            lam = 1.6 / (2.6 ** octave)
            k = 2 * np.pi / lam
            ang = rng.uniform(0, 2 * np.pi, size=10)
            mag = k * rng.uniform(0.7, 1.3, size=10)
            ks.append(np.stack([mag * np.cos(ang), mag * np.sin(ang)], axis=1))
            amps.append(np.full(10, 1.0 / (1.6 ** octave)))
        self.tk = np.concatenate(ks)
        self.ta = np.concatenate(amps)
        self.tp = rng.uniform(0, 2 * np.pi, size=len(self.ta))
        self.tnorm = 2.2 * np.sqrt(0.5 * np.sum(self.ta ** 2))

    def height(self, X, Y):
        h = np.full_like(X, self.z0)
        for (kx, ky), a, p in zip(self.rk, self.ra, self.rp):
            h += a * np.sin(kx * X + ky * Y + p)
        return h

    def height_grad(self, X, Y):
        gx = np.zeros_like(X)
        gy = np.zeros_like(X)
        for (kx, ky), a, p in zip(self.rk, self.ra, self.rp):
            c = a * np.cos(kx * X + ky * Y + p)
            gx += kx * c
            gy += ky * c
        return gx, gy

    def texture(self, X, Y):
        t = np.zeros_like(X)
        for (kx, ky), a, p in zip(self.tk, self.ta, self.tp):
            t += a * np.sin(kx * X + ky * Y + p)
        return 0.5 + 0.5 * np.clip(t / self.tnorm, -1.0, 1.0)  # 0..1

    def render(self, T_wc: np.ndarray, rows: int, cols: int, intr):
        fx, fy, cx, cy = intr
        R, t = T_wc[:3, :3], T_wc[:3, 3]
        r, c = np.meshgrid(np.arange(rows, dtype=np.float64), np.arange(cols, dtype=np.float64), indexing="ij")
        dc = np.stack([(c - cx) / fx, (r - cy) / fy, np.ones_like(c)], axis=-1)
        d = dc @ R.T
        s = np.full((rows, cols), (self.z0 - t[2]))
        for _ in range(8):
            X = t[0] + s * d[..., 0]
            Y = t[1] + s * d[..., 1]
            g = t[2] + s * d[..., 2] - self.height(X, Y)
            hx, hy = self.height_grad(X, Y)
            gp = d[..., 2] - hx * d[..., 0] - hy * d[..., 1]
            s = s - g / gp
        X = t[0] + s * d[..., 0]
        Y = t[1] + s * d[..., 1]
        return self.texture(X, Y), s  # camera-frame depth == s because d_cam.z == 1

    def render_bracketed(self, T_wc: np.ndarray, rows: int, cols: int, intr, steps: int = 48, bisections: int = 24):
        """render() for cameras that look at the height field obliquely. There the straight-down Newton start of render()
        diverges (a grazing ray meets relief slopes where the Newton step overshoots to another branch: residuals of
        kilometres after 40 steps at a 20 degree tilt). Instead the ray is marched through the relief band
        [z0 - 0.5, z0 + 0.5] m to the first sign change of ray z - height (the visible surface), the bracket is bisected and
        three Newton steps polish the root. Returns (texture, depth, largest |ray z - height| in metres)."""
        fx, fy, cx, cy = intr
        R, t = T_wc[:3, :3], T_wc[:3, 3]
        r, c = np.meshgrid(np.arange(rows, dtype=np.float64), np.arange(cols, dtype=np.float64), indexing="ij")
        dc = np.stack([(c - cx) / fx, (r - cy) / fy, np.ones_like(c)], axis=-1)
        d = dc @ R.T
        if np.any(d[..., 2] <= 0.05):
            raise ValueError("a ray does not descend towards the height field")

        def g(s):
            return t[2] + s * d[..., 2] - self.height(t[0] + s * d[..., 0], t[1] + s * d[..., 1])

        s_lo = (self.z0 - 0.5 - t[2]) / d[..., 2]
        s_hi = (self.z0 + 0.5 - t[2]) / d[..., 2]
        a, b = s_lo.copy(), s_hi.copy()
        found = np.zeros(a.shape, dtype=bool)
        prev = s_lo
        for i in range(1, steps + 1):
            cur = s_lo + (s_hi - s_lo) * (i / steps)
            hit = ~found & (g(cur) >= 0)
            a[hit], b[hit] = prev[hit], cur[hit]
            found |= hit
            prev = cur
        for _ in range(bisections):
            m = 0.5 * (a + b)
            up = g(m) >= 0
            b = np.where(up, m, b)
            a = np.where(up, a, m)
        s = 0.5 * (a + b)
        for _ in range(3):
            X = t[0] + s * d[..., 0]
            Y = t[1] + s * d[..., 1]
            hx, hy = self.height_grad(X, Y)
            s = s - g(s) / (d[..., 2] - hx * d[..., 0] - hy * d[..., 1])
        res = float(np.max(np.abs(g(s))))
        return self.texture(t[0] + s * d[..., 0], t[1] + s * d[..., 1]), s, res


def make_pair(seed: int = 1000, rows: int = 480, cols: int = 640, gamma: float = 0.6, gain: float = 0.8,
              bias: float = 0.1, invalid_depth_frac: float = 0.0, motion_scale: float = 1.0) -> Pair:
    """Pair `p` of the benchmark uses seed 1000+p (BASELINE.md section 4)."""
    rng = np.random.default_rng(seed)
    scale = cols / 640.0
    intr4 = (FX * scale, FY * scale, (CX + 0.5) * scale - 0.5, (CY + 0.5) * scale - 0.5)
    scene = _Scene(rng)
    T0 = np.eye(4)
    T0[:3, :3] = _rot(*rng.uniform(-0.02, 0.02, size=3))
    T0[:3, 3] = rng.uniform(-0.05, 0.05, size=3)
    dT = np.eye(4)
    dT[:3, :3] = _rot(*(rng.uniform(-0.01, 0.01, size=3) * motion_scale))
    dT[:3, 3] = rng.uniform(-0.02, 0.02, size=3) * motion_scale
    T1 = T0 @ dT
    tex0, z0 = scene.render(T0, rows, cols, intr4)
    tex1, _ = scene.render(T1, rows, cols, intr4)
    im0 = np.clip(np.rint(255.0 * tex0), 0, 255).astype(np.uint8)
    lit = gain * np.power(tex1, gamma) + bias
    im1 = np.clip(np.rint(255.0 * lit), 0, 255).astype(np.uint8)
    d16 = np.clip(np.rint(z0 * 5000.0), 0, 65535).astype(np.uint16)
    if invalid_depth_frac > 0:
        mask = rng.uniform(size=d16.shape) < invalid_depth_frac
        d16[mask] = 0
    depth = d16.astype(np.float64) * DEPTH_FACTOR
    intr = np.array([*intr4, DEPTH_FACTOR], dtype=np.float64)
    return Pair(im0=im0, im1=im1, depth0=depth, depth0_u16=d16,
                T_wc0=np.ascontiguousarray(T0.T).reshape(16).copy(),
                T_wc1=np.ascontiguousarray(T1.T).reshape(16).copy(),
                intr=intr, rows=rows, cols=cols)


def make_sequence(seed: int, n: int, rows: int = 480, cols: int = 640) -> list:
    """n distinct pairs that share one rendered scene (two ray-cast frames, ~1.5 s at 640x480) and differ in what a
    tracking sequence varies cheaply: pair k sees its own exposure of the reference frame (gain/bias before the 8-bit
    quantisation), its own gamma/affine illumination change of the target frame, so every pair has its own im0 (and
    with it its own reference classes), its own im1 and its own solution; depth and ground-truth poses are the
    scene's. Pair 0 is make_pair(seed) itself. Used for BASELINE config 4 (1024 pairs = 16 scenes x 64 pairs)."""
    rng = np.random.default_rng(seed)
    scale = cols / 640.0
    intr4 = (FX * scale, FY * scale, (CX + 0.5) * scale - 0.5, (CY + 0.5) * scale - 0.5)
    scene = _Scene(rng)
    T0 = np.eye(4)
    T0[:3, :3] = _rot(*rng.uniform(-0.02, 0.02, size=3))
    T0[:3, 3] = rng.uniform(-0.05, 0.05, size=3)
    dT = np.eye(4)
    dT[:3, :3] = _rot(*rng.uniform(-0.01, 0.01, size=3))
    dT[:3, 3] = rng.uniform(-0.02, 0.02, size=3)
    T1 = T0 @ dT
    tex0, z0 = scene.render(T0, rows, cols, intr4)
    tex1, _ = scene.render(T1, rows, cols, intr4)
    d16 = np.clip(np.rint(z0 * 5000.0), 0, 65535).astype(np.uint16)
    depth = d16.astype(np.float64) * DEPTH_FACTOR
    intr = np.array([*intr4, DEPTH_FACTOR], dtype=np.float64)
    vr = np.random.default_rng(seed * 7919 + 13)
    out = []
    for k in range(n):
        if k == 0:
            a0, b0, gamma, gain, bias = 1.0, 0.0, 0.6, 0.8, 0.1
        else:
            a0, b0 = vr.uniform(0.85, 1.0), vr.uniform(0.0, 0.08)
            gamma, gain, bias = vr.uniform(0.45, 1.2), vr.uniform(0.7, 0.95), vr.uniform(0.0, 0.12)
        im0 = np.clip(np.rint(255.0 * (a0 * tex0 + b0)), 0, 255).astype(np.uint8)
        im1 = np.clip(np.rint(255.0 * (gain * np.power(tex1, gamma) + bias)), 0, 255).astype(np.uint8)
        out.append(Pair(im0=im0, im1=im1, depth0=depth, depth0_u16=d16,
                        T_wc0=np.ascontiguousarray(T0.T).reshape(16).copy(),
                        T_wc1=np.ascontiguousarray(T1.T).reshape(16).copy(), intr=intr, rows=rows, cols=cols))
    return out


def mat16_inverse(m16: np.ndarray) -> np.ndarray:
    """Rigid inverse of a column-major 4x4."""
    M = m16.reshape(4, 4).T
    Rm, t = M[:3, :3], M[:3, 3]
    Mi = np.eye(4)
    Mi[:3, :3] = Rm.T
    Mi[:3, 3] = -Rm.T @ t
    return np.ascontiguousarray(Mi.T).reshape(16).copy()


# largest |ray z - height| (metres) a frame of the multi-view generators below may leave; checked on every render
RENDER_TOL = 1e-9


def _render_checked(scene: _Scene, T_wc, rows, cols, intr4):
    tex, z, res = scene.render_bracketed(T_wc, rows, cols, intr4)
    if not res < RENDER_TOL:
        raise RuntimeError(f"ray cast did not converge: residual {res:.3g} m")
    return tex, z


def _col16(T: np.ndarray) -> np.ndarray:
    return np.ascontiguousarray(T.T).reshape(16).copy()


def _pair_from(tex0, z0, tex1, T0, T1, intr4, rows, cols, expo0=(1.0, 0.0), light1=(0.6, 0.8, 0.1)) -> Pair:
    a0, b0 = expo0
    gamma, gain, bias = light1
    im0 = np.clip(np.rint(255.0 * (a0 * tex0 + b0)), 0, 255).astype(np.uint8)
    im1 = np.clip(np.rint(255.0 * (gain * np.power(tex1, gamma) + bias)), 0, 255).astype(np.uint8)
    d16 = np.clip(np.rint(z0 * 5000.0), 0, 65535).astype(np.uint16)
    return Pair(im0=im0, im1=im1, depth0=d16.astype(np.float64) * DEPTH_FACTOR, depth0_u16=d16, T_wc0=_col16(T0),
                T_wc1=_col16(T1), intr=np.array([*intr4, DEPTH_FACTOR], dtype=np.float64), rows=rows, cols=cols)


@dataclasses.dataclass
class Rig:
    pairs: list            # pair g: camera g at the reference body pose -> camera g at the target body pose
    T_cb: np.ndarray       # float64 [n_cams, 16] column-major camera-from-body; camera 0 is the body (identity)
    T_wb0: np.ndarray      # float64 [16] body-to-world, reference
    T_wb1: np.ndarray      # float64 [16] body-to-world, target (the ground truth of a rig solve is its inverse)


def make_rig(seed: int, n_cams: int, rows: int = 480, cols: int = 640, motion_scale: float = 1.0) -> Rig:
    """A rigid multi-camera rig over one scene: one body motion (as make_pair draws a camera motion) seen by n_cams cameras.
    Camera 0 is the body frame; camera g >= 1 is tilted by 15-25 degrees about x and y (alternating signs, so that the
    views point different ways) and offset by a few centimetres. Every camera renders both body poses exactly."""
    rng = np.random.default_rng(seed)
    scale = cols / 640.0
    intr4 = (FX * scale, FY * scale, (CX + 0.5) * scale - 0.5, (CY + 0.5) * scale - 0.5)
    scene = _Scene(rng)
    Tb0 = np.eye(4)
    Tb0[:3, :3] = _rot(*rng.uniform(-0.02, 0.02, size=3))
    Tb0[:3, 3] = rng.uniform(-0.05, 0.05, size=3)
    dT = np.eye(4)
    dT[:3, :3] = _rot(*(rng.uniform(-0.01, 0.01, size=3) * motion_scale))
    dT[:3, 3] = rng.uniform(-0.02, 0.02, size=3) * motion_scale
    Tb1 = Tb0 @ dT
    pairs, T_cb = [], []
    for g in range(n_cams):
        T_bc = np.eye(4)
        if g > 0:
            tilt = np.deg2rad(rng.uniform(15.0, 25.0, size=2)) * np.array([(-1) ** g, (-1) ** (g // 2)])
            T_bc[:3, :3] = _rot(tilt[0], tilt[1], rng.uniform(-0.1, 0.1))
            T_bc[:3, 3] = rng.uniform(-0.05, 0.05, size=3)
        T0, T1 = Tb0 @ T_bc, Tb1 @ T_bc
        tex0, z0 = _render_checked(scene, T0, rows, cols, intr4)
        tex1, _ = _render_checked(scene, T1, rows, cols, intr4)
        pairs.append(_pair_from(tex0, z0, tex1, T0, T1, intr4, rows, cols))
        T_cb.append(mat16_inverse(_col16(T_bc)))
    return Rig(pairs=pairs, T_cb=np.stack(T_cb), T_wb0=_col16(Tb0), T_wb1=_col16(Tb1))


def make_keyframes(seed: int, n_refs: int, rows: int = 480, cols: int = 640, motion_scale: float = 1.0) -> list:
    """n_refs reference keyframes of one target frame: pair k has reference frame k (its own pose, drawn as make_pair draws
    a motion, and its own exposure) and the common target frame, so every pair has the same im1 and T_wc1."""
    rng = np.random.default_rng(seed)
    scale = cols / 640.0
    intr4 = (FX * scale, FY * scale, (CX + 0.5) * scale - 0.5, (CY + 0.5) * scale - 0.5)
    scene = _Scene(rng)
    T1 = np.eye(4)
    T1[:3, :3] = _rot(*rng.uniform(-0.02, 0.02, size=3))
    T1[:3, 3] = rng.uniform(-0.05, 0.05, size=3)
    tex1, _ = _render_checked(scene, T1, rows, cols, intr4)
    pairs = []
    for k in range(n_refs):
        dT = np.eye(4)
        dT[:3, :3] = _rot(*(rng.uniform(-0.02, 0.02, size=3) * motion_scale))
        dT[:3, 3] = rng.uniform(-0.04, 0.04, size=3) * motion_scale
        T0 = T1 @ dT
        tex0, z0 = _render_checked(scene, T0, rows, cols, intr4)
        expo = (rng.uniform(0.85, 1.0), rng.uniform(0.0, 0.08)) if k > 0 else (1.0, 0.0)
        pairs.append(_pair_from(tex0, z0, tex1, T0, T1, intr4, rows, cols, expo0=expo))
    return pairs
