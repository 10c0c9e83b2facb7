"""Synthetic 8-bit grayscale inputs for the feature front end (SURVEY.md 8d "Input hygiene").

Every frame is generated ONCE as bytes (numpy, seeded) and the identical buffer is handed to the
CUDA path and to the checker, so generator floating-point details never enter a parity claim.

  blob_pair / blob_quad ... generator (A): background 96 plus Gaussian blobs, second frame = the same
                            field shifted by a few pixels (flow), right camera = shifted by a disparity.
  corridor_frame .......... generator (B): pin-hole ray cast of a textured corridor (floor, ceiling, two
                            walls) with real depth structure, needed by the mono odometry configs because
                            pure image-plane translations make the 8-point problem degenerate.
"""
import numpy as np

KITTI_F, KITTI_CU, KITTI_CV = 645.2, 635.9, 194.1   # matlab/demo_viso_mono.m:9-11 of the reference


def _blob_canvas(width, height, n_blobs, seed, margin):
    rng = np.random.default_rng(seed)
    W, H = width + 2 * margin, height + 2 * margin
    canvas = np.full((H, W), 96.0, dtype=np.float32)
    cx = rng.uniform(0, W, n_blobs)
    cy = rng.uniform(0, H, n_blobs)
    sig = rng.uniform(2.0, 7.0, n_blobs)
    amp = rng.uniform(-130.0, 130.0, n_blobs)
    for i in range(n_blobs):
        r = int(3 * sig[i]) + 1
        x0, x1 = max(int(cx[i]) - r, 0), min(int(cx[i]) + r + 1, W)
        y0, y1 = max(int(cy[i]) - r, 0), min(int(cy[i]) + r + 1, H)
        if x0 >= x1 or y0 >= y1:
            continue
        xs = np.arange(x0, x1, dtype=np.float32) - np.float32(cx[i])
        ys = np.arange(y0, y1, dtype=np.float32) - np.float32(cy[i])
        g = np.exp(-(ys[:, None] ** 2 + xs[None, :] ** 2) / np.float32(2 * sig[i] ** 2))
        canvas[y0:y1, x0:x1] += np.float32(amp[i]) * g
    return canvas


def _crop(canvas, width, height, margin, dx, dy):
    x0, y0 = margin + dx, margin + dy
    return np.clip(np.rint(canvas[y0:y0 + height, x0:x0 + width]), 0, 255).astype(np.uint8)


def default_blob_count(width, height):
    return int(round(6000 * (width * height) / (1241.0 * 376.0)))


def blob_pair(width=1241, height=376, n_blobs=None, seed=1234, shift=(3, 1)):
    """Two frames of the same blob field; the second is the field shifted by `shift` pixels."""
    if n_blobs is None:
        n_blobs = default_blob_count(width, height)
    m = 100
    c = _blob_canvas(width, height, n_blobs, seed, m)
    return _crop(c, width, height, m, 0, 0), _crop(c, width, height, m, -shift[0], -shift[1])


def blob_quad(width=1241, height=376, n_blobs=None, seed=1234, shift=(3, 1), disparity=12):
    """(left_prev, right_prev, left_curr, right_curr); the right camera sees the field shifted by -disparity."""
    if n_blobs is None:
        n_blobs = default_blob_count(width, height)
    m = 100
    c = _blob_canvas(width, height, n_blobs, seed, m)
    lp = _crop(c, width, height, m, 0, 0)
    rp = _crop(c, width, height, m, disparity, 0)
    lc = _crop(c, width, height, m, -shift[0], -shift[1])
    rc = _crop(c, width, height, m, -shift[0] + disparity, -shift[1])
    return lp, rp, lc, rc


def blob_sequence(n_frames, width=1241, height=376, n_blobs=None, seed=1234, step=(3, 1)):
    """n_frames crops of one blob field, each shifted by `step` from the last (flow benchmark input)."""
    if n_blobs is None:
        n_blobs = default_blob_count(width, height)
    m = 100
    c = _blob_canvas(width, height, n_blobs, seed, m)
    out = np.empty((n_frames, height, width), dtype=np.uint8)
    for k in range(n_frames):
        dx = (k * step[0]) % (2 * m - 2) - (m - 1)
        dy = (k * step[1]) % (2 * m - 2) - (m - 1)
        out[k] = _crop(c, width, height, m, -dx, -dy)
    return out


# ----------------------------------------------------------------------------- corridor ray cast
def _hash01(ix, iy, seed):
    h = (ix.astype(np.uint32) * np.uint32(73856093)) ^ (iy.astype(np.uint32) * np.uint32(19349663)) ^ np.uint32((seed * 83492791) & 0xFFFFFFFF)
    h ^= h >> np.uint32(13)
    h *= np.uint32(0x5BD1E995)
    h ^= h >> np.uint32(15)
    return (h & np.uint32(0xFFFF)).astype(np.float32) / np.float32(65535.0)


def _value_noise(x, y, seed, octaves=4, base=2.0, lacunarity=2.3, gain=0.6):
    total = np.zeros_like(x, dtype=np.float32)
    amp, freq, norm = 1.0, base, 0.0
    for o in range(octaves):
        fx, fy = x * np.float32(freq), y * np.float32(freq)
        ix, iy = np.floor(fx), np.floor(fy)
        tx, ty = fx - ix, fy - iy
        tx = tx * tx * (3 - 2 * tx)
        ty = ty * ty * (3 - 2 * ty)
        ix, iy = ix.astype(np.int64), iy.astype(np.int64)
        v00 = _hash01(ix, iy, seed + 17 * o)
        v10 = _hash01(ix + 1, iy, seed + 17 * o)
        v01 = _hash01(ix, iy + 1, seed + 17 * o)
        v11 = _hash01(ix + 1, iy + 1, seed + 17 * o)
        total += np.float32(amp) * ((v00 * (1 - tx) + v10 * tx) * (1 - ty) + (v01 * (1 - tx) + v11 * tx) * ty)
        norm += amp
        amp *= gain
        freq *= lacunarity
    return total / np.float32(norm)


def _corridor_rays(k, width, height, f, cu, cv, cam_height, pitch, step, baseline_x):
    """Ray cast of corridor_frame: per pixel the surface hit (0 floor, 1 ceiling, 2 / 3 walls), the ray parameter t
    (capped at 400) and the hit point."""
    scale = width / 1241.0
    f, cu, cv = f * scale, cu * scale, cv * scale
    u = np.arange(width, dtype=np.float32)[None, :]
    v = np.arange(height, dtype=np.float32)[:, None]
    dx = np.broadcast_to((u - np.float32(cu)) / np.float32(f), (height, width)).astype(np.float32)
    dy = np.broadcast_to((v - np.float32(cv)) / np.float32(f), (height, width)).astype(np.float32)
    dz = np.ones((height, width), dtype=np.float32)
    # pitch about x (negative = looking down), then yaw about y
    cp, sp = np.float32(np.cos(-pitch)), np.float32(np.sin(-pitch))
    dy2 = cp * dy + sp * dz
    dz2 = -sp * dy + cp * dz
    yaw = 0.01 * np.sin(0.3 * k)
    cyw, syw = np.float32(np.cos(yaw)), np.float32(np.sin(yaw))
    dx3 = cyw * dx + syw * dz2
    dz3 = -syw * dx + cyw * dz2
    dy3 = dy2
    ox, oy, oz = np.float32(baseline_x), np.float32(0.0), np.float32(step * k)
    big = np.float32(1e9)
    with np.errstate(divide='ignore', invalid='ignore'):
        t_floor = np.where(dy3 > 1e-6, (np.float32(cam_height) - oy) / dy3, big)
        t_ceil = np.where(dy3 < -1e-6, (np.float32(-4.0) - oy) / dy3, big)
        t_wr = np.where(dx3 > 1e-6, (np.float32(6.0) - ox) / dx3, big)
        t_wl = np.where(dx3 < -1e-6, (np.float32(-6.0) - ox) / dx3, big)
    ts = np.stack([t_floor, t_ceil, t_wr, t_wl])
    which = np.argmin(ts, axis=0)
    t = np.min(ts, axis=0)
    t = np.minimum(t, np.float32(400.0))
    px, py, pz = ox + t * dx3, oy + t * dy3, oz + t * dz3
    return which, t, px, py, pz


def corridor_frame(k, width=1241, height=376, seed=1234, f=KITTI_F, cu=KITTI_CU, cv=KITTI_CV,
                   cam_height=1.6, pitch=-0.08, step=0.8, baseline_x=0.0):
    """Frame k of a forward drive (0.8 m per frame, yaw 0.01*sin(0.3k)) through a textured corridor.
    Camera axes: x right, y down, z forward.  Floor y=+cam_height, ceiling y=-4, walls x=+-6."""
    which, t, px, py, pz = _corridor_rays(k, width, height, f, cu, cv, cam_height, pitch, step, baseline_x)
    img = np.zeros((height, width), dtype=np.float32)
    for s, (a, b) in enumerate([(px, pz), (px, pz), (py, pz), (py, pz)]):
        m = which == s
        if m.any():
            img[m] = _value_noise(a[m], b[m], seed * 4 + s)
    fade = np.clip(np.float32(1.0) - t / np.float32(120.0), 0.15, 1.0)
    out = np.float32(128.0) + (img - np.float32(0.5)) * np.float32(330.0) * fade
    return np.clip(np.rint(out), 0, 255).astype(np.uint8)


def corridor_depth(k, width=1241, height=376, f=KITTI_F, cu=KITTI_CU, cv=KITTI_CV, cam_height=1.6, pitch=-0.08, step=0.8,
                   baseline_x=0.0):
    """The ray parameter t of corridor_frame per pixel, (height, width) float32: the depth Z in the camera frame, since
    every ray has dz = 1 there.  t is capped at 400 where the ray leaves the corridor."""
    return _corridor_rays(k, width, height, f, cu, cv, cam_height, pitch, step, baseline_x)[1]


def corridor_sequence(n_frames, width=1241, height=376, seed=1234, start=0, **kw):
    return np.stack([corridor_frame(start + k, width, height, seed, **kw) for k in range(n_frames)])


def corridor_stereo_frame(k, width=1241, height=376, seed=1234, baseline=0.54):
    return corridor_frame(k, width, height, seed), corridor_frame(k, width, height, seed, baseline_x=baseline)


def track_sequence(n_frames=12, n_points=600, seed=11, width=1241, height=376, f=KITTI_F, cu=KITTI_CU, cv=KITTI_CV,
                   step=0.8, drop=0.15, noise=0.2):
    """Synthetic feature tracks for the Reconstruction tests: random 3-D points ahead of a camera that drives forward
    with a slight yaw; every frame pair yields flow matches (48-byte p_match records, only the 1p / 1c fields used)
    whose feature indices chain from frame to frame like the matcher's i1p / i1c, plus the motion previous -> current
    camera frame.  Points drop out at random so that tracks end and get reconstructed.  Returns a list of
    (matches, Tr) per frame pair."""
    rng = np.random.RandomState(seed)
    P = np.stack([rng.uniform(-8, 8, n_points), rng.uniform(-2.5, 1.6, n_points), rng.uniform(4, 60, n_points)], 1)
    dt = np.dtype([('u1p', 'f4'), ('v1p', 'f4'), ('i1p', 'i4'), ('u2p', 'f4'), ('v2p', 'f4'), ('i2p', 'i4'),
                   ('u1c', 'f4'), ('v1c', 'f4'), ('i1c', 'i4'), ('u2c', 'f4'), ('v2c', 'f4'), ('i2c', 'i4')])
    poses = []                      # world -> camera k
    for k in range(n_frames):
        yaw = 0.01 * np.sin(0.3 * k)
        R = np.array([[np.cos(yaw), 0, -np.sin(yaw)], [0, 1, 0], [np.sin(yaw), 0, np.cos(yaw)]])
        T = np.eye(4); T[:3, :3] = R; T[:3, 3] = -R @ np.array([0.05 * k, 0.0, step * k])
        poses.append(T)
    obs = []
    for k in range(n_frames):
        X = P @ poses[k][:3, :3].T + poses[k][:3, 3]
        u = f * X[:, 0] / X[:, 2] + cu + rng.normal(0, noise, n_points)
        v = f * X[:, 1] / X[:, 2] + cv + rng.normal(0, noise, n_points)
        vis = (X[:, 2] > 1.5) & (u > 6) & (u < width - 7) & (v > 6) & (v < height - 7) & (rng.rand(n_points) > drop)
        index = rng.permutation(n_points).astype(np.int32)          # feature index of every point in this frame
        obs.append((u.astype(np.float32), v.astype(np.float32), vis, index))
    out = []
    for k in range(1, n_frames):
        up, vp, visp, ip = obs[k - 1]
        uc, vc, visc, ic = obs[k]
        both = np.nonzero(visp & visc)[0]
        both = both[np.argsort(ic[both])]
        m = np.zeros(len(both), dt)
        for name in ('u2p', 'v2p', 'u2c', 'v2c'):
            m[name] = -1
        m['i2p'] = -1; m['i2c'] = -1
        m['u1p'] = up[both]; m['v1p'] = vp[both]; m['i1p'] = ip[both]
        m['u1c'] = uc[both]; m['v1c'] = vc[both]; m['i1c'] = ic[both]
        out.append((m, poses[k] @ np.linalg.inv(poses[k - 1])))
    return out
