"""Pins the CPU oracle's tracking half against the REFERENCE's own CUDA kernels and checks the product against the same
reference outputs. tests/golden/ref_pin_640x480.npz holds what the reference's reduce.cu and cudafuncs.cu (compiled unmodified,
oracle/ref_harness.cu driving them) computed on a B200 from the inputs below (generator: tests/golden/make_ref_pin_golden.py):
pyramid NaN masks in full, map values at a fixed seeded sample of pixels, ICP steps and the whole tracking run in full.
Tolerances cover what legitimately differs: nvcc's FMA contraction and approximate rsqrtf in the reference build vs single
IEEE ops in oracle/product, and reduction order."""
import os

import numpy as np
import pytest

from util import digest, pose_inputs, rel_err, tracking_inputs

pytestmark = pytest.mark.gpu

LEVELS = (0, 1, 2)
G_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_pin_640x480.npz")


@pytest.fixture(scope="module")
def rstate(frames, K):
    from oracle import ef_oracle as eo

    g = dict(np.load(G_PATH))
    x = tracking_inputs(frames, K)
    assert digest(x) == str(g["inputs_sha256"]), "the tracking inputs changed: regenerate tests/golden/ref_pin_640x480.npz"
    od = eo.Odometry(K.width, K.height, K.cx, K.cy, K.fx, K.fy)
    od.init_first_rgb(x["prev_rgba"])  # previous live frame -> lastNextImage, as the pipeline had it
    od.init_icp_model(x["vtx"], x["nrm"], x["T"])
    od.init_rgb_model(x["img"])
    od.init_icp_depth(x["filt"], 20.0)
    od.init_rgb(x["rgba"])
    return dict(g=g, x=x, od=od, T=x["T"], K=K)


def _cmp_map(a, g, name, lv, tol):
    """a: the oracle's (3 rows, cols) map; g: the reference's NaN mask of the x plane, sampled values, sums and magnitude."""
    planes = a.reshape(3, -1)
    av = ~np.isnan(planes[0])
    bv = ~np.unpackbits(g[f"{name}{lv}_nan"])[:av.size].astype(bool)
    assert (av != bv).mean() < 1e-4, f"{name}{lv}: validity differs on {(av != bv).mean():.2e} of the pixels"
    idx, q = g[f"idx{lv}"], g[f"{name}{lv}_s"]
    p = planes[:, idx]
    m = av[idx] & bv[idx]
    assert m.sum() > 0.3 * len(idx), name
    s, s_abs, q_max = g[f"{name}{lv}_stats"]
    assert np.abs(p[:, m] - q[:, m]).max() <= tol * max(1.0, q_max), f"{name}{lv}"
    ok = av & bv
    v = planes[:, ok].astype(np.float64)
    assert abs(np.abs(v).sum() - s_abs) <= 2e-4 * s_abs and abs(v.sum() - s) <= 2e-4 * s_abs, (name, lv, v.sum(), s)


@pytest.mark.parametrize("lv", LEVELS)
def test_oracle_pyramids_match_reference_kernels(rstate, lv):
    od, g = rstate["od"], rstate["g"]
    assert digest({"a": od.buffer("depth_tmp", lv)}) == str(g[f"depth_tmp{lv}_sha256"])
    _cmp_map(od.buffer("vmap_curr", lv), g, "vmap_curr", lv, 1e-6)
    _cmp_map(od.buffer("nmap_curr", lv), g, "nmap_curr", lv, 2e-6)
    _cmp_map(od.buffer("vmap_g_prev", lv), g, "vmap_g_prev", lv, 1e-6)
    _cmp_map(od.buffer("nmap_g_prev", lv), g, "nmap_g_prev", lv, 2e-6)
    idx = g[f"idx{lv}"]
    for n in ("lastDepth", "nextDepth"):
        a = od.buffer(n, lv).reshape(-1)
        assert np.array_equal(np.isnan(a), np.unpackbits(g[f"{n}{lv}_nan"])[:a.size].astype(bool)), n
        assert np.nanmax(np.abs(a[idx] - g[f"{n}{lv}_s"])) <= 2e-6, n
    for n in ("lastImage", "nextImage", "lastNextImage"):
        a, b = od.buffer(n, lv).reshape(-1)[idx].astype(int), g[f"{n}{lv}_s"].astype(int)
        # int(0.114 x + 0.299 y + 0.587 z): FMA contraction can move a value across an integer boundary
        assert np.abs(a - b).max() <= 1 and (a != b).mean() < 2e-3, (n, (a != b).mean())


@pytest.mark.parametrize("lv", LEVELS)
def test_oracle_icp_step_matches_reference_icpStep(rstate, lv):
    from oracle import ef_oracle as eo

    od, g, K = rstate["od"], rstate["g"], rstate["K"]
    Rc, tc, Rpi, tp = pose_inputs(rstate["T"])
    d = np.float32(1 << lv)
    ang = float(np.sin(np.float32(20.0) * np.float32(3.14159254) / np.float32(180.0)))
    # the oracle's own maps, which the pyramid test above pins to the reference's maps
    Ao, bo, ro = eo.icp_step(Rc, tc, od.buffer("vmap_curr", lv), od.buffer("nmap_curr", lv), Rpi, tp, np.float32(K.fx) / d, np.float32(K.fy) / d,
                             np.float32(K.cx) / d, np.float32(K.cy) / d, od.buffer("vmap_g_prev", lv), od.buffer("nmap_g_prev", lv), 0.10, ang)
    Ar, br, rr = g[f"icp_A{lv}"], g[f"icp_b{lv}"], g[f"icp_r{lv}"]
    assert abs(rr[1] - ro[1]) <= max(2, 2e-4 * ro[1]), (rr[1], ro[1])
    assert rel_err(Ao, Ar) < 2e-4 and rel_err(bo, br) < 2e-4 and abs(ro[0] - rr[0]) < 2e-4 * rr[0]


def _ref_trace(g):
    from oracle import ef_oracle as eo

    return g["track_T"], g["track_trace"].view(eo.TRACE_DTYPE)


def test_oracle_track_matches_reference_track(rstate):
    """Whole getIncrementalTransformation: oracle host loop + oracle kernels vs harness host loop (Eigen) + reference kernels."""
    od, T = rstate["od"], rstate["T"]
    To, tro = od.track(T)
    Tr, trr = _ref_trace(rstate["g"])
    assert len(tro) == len(trr)
    for a, b in zip(tro, trr):
        assert (a["kind"], a["level"], a["iter"]) == (b["kind"], b["level"], b["iter"])
        if a["kind"] == 0:
            assert rel_err(a["lastA"], b["lastA"]) < 2e-3, (a["level"], a["iter"], rel_err(a["lastA"], b["lastA"]))
    assert np.abs(To[:3, 3] - Tr[:3, 3]).max() < 2e-5 and np.abs(To[:3, :3] - Tr[:3, :3]).max() < 2e-5


def test_product_track_matches_reference_track(K, rstate):
    """The product (device-resident GN loop) against the reference kernels driven like the reference: per-iteration
    JtJ/Jtr and the final pose (BASELINE.json: 1e-4 relative on identical inputs; the chained loop is looser, see
    test_gpu_tracking.py)."""
    from elasticfusion_b200 import capi

    x, g, T = rstate["x"], rstate["g"], rstate["T"]
    ctx = capi.Context(capi.default_config(K.width, K.height, K.fx, K.fy, K.cx, K.cy, capacity=400000))
    try:
        ctx.upload("FILL_VERTEX", x["vtx"])
        ctx.upload("FILL_NORMAL", x["nrm"])
        ctx.upload("FILL_IMAGE", x["img"])
        ctx.upload("DEPTH_FILTERED", x["filt"])
        ctx.upload("RGBA", x["prev_rgba"])
        ctx.odom_init_first_rgb(ctx.buffer_ptr("RGBA")[0])
        ctx.upload("RGBA", x["rgba"])
        ctx.odom_init_icp_model(ctx.buffer_ptr("FILL_VERTEX")[0], ctx.buffer_ptr("FILL_NORMAL")[0], T)
        ctx.odom_init_rgb_model(ctx.buffer_ptr("FILL_IMAGE")[0])
        ctx.odom_init_icp_depth(ctx.buffer_ptr("DEPTH_FILTERED")[0], 20.0)
        ctx.odom_init_rgb(ctx.buffer_ptr("RGBA")[0])
        # identical-input single step first
        Rc, tc, Rpi, tp = pose_inputs(T)
        Ap, bp, rp = ctx.icp_step(0, Rc, tc, Rpi, tp)
        Ar, br = g["icp_A0"], g["icp_b0"]
        assert rel_err(Ap, Ar) < 3e-4 and rel_err(bp, br) < 3e-4, (rel_err(Ap, Ar), rel_err(bp, br))
        Tp, trp = ctx.odom_track(T)
        Tr, trr = _ref_trace(g)
        assert len(trp) == len(trr)
        assert np.abs(Tp[:3, 3] - Tr[:3, 3]).max() < 2e-5 and np.abs(Tp[:3, :3] - Tr[:3, :3]).max() < 2e-5
    finally:
        ctx.close()
