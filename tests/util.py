"""Shared helpers for the parity tests."""
import numpy as np


def rgba_of(rgb):
    h, w, _ = rgb.shape
    return np.ascontiguousarray(np.concatenate([rgb, np.full((h, w, 1), 255, np.uint8)], -1))


def assert_same(a, b, what=""):
    """Bit-exact, NaN-aware equality."""
    a = np.asarray(a)
    b = np.asarray(b)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    if a.dtype.kind == "f":
        ok = (a == b) | (np.isnan(a) & np.isnan(b))
    else:
        ok = a == b
    if a.dtype.names:
        ok = np.ones(a.shape, bool)
        for n in a.dtype.names:
            ok &= (a[n] == b[n]) | ((a[n] != a[n]) & (b[n] != b[n]))
    bad = int((~ok).sum())
    assert bad == 0, f"{what}: {bad} of {ok.size} elements differ"


def valid_planes(m):
    """SoA 3-plane map -> (x,y,z planes, valid mask from the x plane)."""
    r = m.shape[0] // 3
    x, y, z = m[:r], m[r:2 * r], m[2 * r:]
    return x, y, z, ~np.isnan(x)


def assert_same_map(a, b, what=""):
    """The reference flags invalid map entries by NaN in the x plane only (y/z stale): compare validity + valid values."""
    ax, ay, az, av = valid_planes(a)
    bx, by, bz, bv = valid_planes(b)
    assert np.array_equal(av, bv), f"{what}: validity differs at {(av != bv).sum()} pixels"
    for p, q, n in ((ax, bx, "x"), (ay, by, "y"), (az, bz, "z")):
        bad = int((p[av] != q[av]).sum())
        assert bad == 0, f"{what}.{n}: {bad} valid values differ"


def rel_err(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def run_oracle(frames, K, n, **kw):
    """Runs the CPU oracle pipeline over the first n frames; returns the Fusion object."""
    from oracle import ef_oracle as eo

    f = eo.Fusion(K, **kw)
    for i in range(n):
        f.process_frame(frames[i][0], frames[i][1], i * 33333)
    return f


def tracking_inputs(frames, K):
    """The inputs of one tracking step after three frames of the CPU oracle: frame 3's filtered depth and colour, frame 2's
    colour, the oracle's pose and fill-in model maps (vertex, normal, image)."""
    from oracle import ef_oracle as eo

    f = run_oracle(frames, K, 3)
    return dict(filt=eo.bilateral(frames[3][1], 3.0), rgba=rgba_of(frames[3][0]), prev_rgba=rgba_of(frames[2][0]), T=f.pose,
                vtx=f.buffer("fill_vertex"), nrm=f.buffer("fill_normal"), img=f.buffer("fill_image"))


def pose_inputs(T):
    """Rcurr, tcurr, Rprev^-1, tprev of one ICP step: the pose T moved by a small rotation and translation."""
    R = T[:3, :3].astype(np.float32)
    t = T[:3, 3].astype(np.float32)
    dR = np.array([[1, -0.002, 0.001], [0.002, 1, -0.003], [-0.001, 0.003, 1]], np.float32)
    return (R @ dR).astype(np.float32), t + np.array([0.004, -0.003, 0.005], np.float32), np.linalg.inv(R).astype(np.float32), t


def digest(arrays):
    """sha256 over the names, shapes, dtypes and bytes of a dict of arrays."""
    import hashlib

    h = hashlib.sha256()
    for k in sorted(arrays):
        a = np.ascontiguousarray(arrays[k])
        h.update(f"{k}{a.shape}{a.dtype.str}".encode())
        h.update(a.tobytes())
    return h.hexdigest()


def oracle_sensitivity(frames, K, **cfg):
    """How far the ORACLE moves from itself when one depth pixel of frame 1 is 1 mm deeper: the scale below which a
    trajectory difference says nothing about an implementation (tracking amplifies any rounding difference the same way).
    Returns (oracle poses of the unperturbed run, ATE RMSE between the two runs, largest per-frame |dT| element)."""
    from elasticfusion_b200 import synth

    runs = []
    for perturb in (False, True):
        f = run_oracle(frames, K, 0, **cfg)
        est = []
        for i, fr in enumerate(frames):
            d = fr[1]
            if perturb and i == 1:
                d = d.copy()
                d[K.height // 2, K.width // 2] += 1
            f.process_frame(fr[0], d, i * 33333)
            est.append(f.pose.copy())
        runs.append(np.array(est))
    return runs[0], float(synth.ate_rmse(runs[0], runs[1])), float(np.abs(runs[0] - runs[1]).max())
