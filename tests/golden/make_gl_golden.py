"""Generates the fixtures of tests/test_gl_golden.py: the inputs and outputs of every GLSL pass of the reference's mapping half,
produced by the REFERENCE's OWN SHADER FILES (its Core/Shaders, unmodified) executed on Mesa llvmpipe through
oracle/gl/ref_gl_harness.cpp (`make -C oracle refgl`). Run where the reference tree and that Mesa build are present:

    python tests/golden/make_gl_golden.py            tests/golden/ref_mapping_160x120.npz: the default camera, every array in full
    python tests/golden/make_gl_golden.py --live     tests/golden/ref_mapping_live.npz: three more cameras (LIVE_CONFIGS), sampled
    python tests/golden/make_gl_golden.py --check C  compares the oracle with the shaders' outputs in configuration C, writes nothing

The chain of inputs is the one a frame goes through (the stage outputs of the CPU oracle feed the next stage on both sides, so
every pass is compared on identical inputs); `gl_*` arrays are what the reference's shaders computed. The live fixture stores no
inputs (tests/test_gl_golden.py regenerates them with inputs() and checks their digest) and, of every shader output, a fixed
strided sample: the pixels of PIXELS() and the surfel rows of ROWS() together with the full row count."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from elasticfusion_b200 import synth  # noqa: E402
from oracle import ef_oracle as eo  # noqa: E402
from util import digest, run_oracle  # noqa: E402

MAXD, BIG = 20.0, 2 ** 30
LIVE_PATH = os.path.join(ROOT, "tests", "golden", "ref_mapping_live.npz")
PIXEL_STRIDE = 41  # prime: the sample walks diagonally across the image rows
ROW_SAMPLE = 512  # surfel rows per list


def graph_for(m, n_nodes=40, seed=4):
    rng = np.random.RandomState(seed)
    idx = np.sort(rng.choice(len(m), n_nodes, replace=False))
    nodes = np.zeros((n_nodes, 16), np.float32)
    for k, i in enumerate(idx):
        w = rng.standard_normal(3) * 0.01
        th = np.linalg.norm(w)
        kx = np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]]) / max(th, 1e-12)
        R = np.eye(3) + np.sin(th) * kx + (1 - np.cos(th)) * (kx @ kx)
        nodes[k, 0:3] = m[i, 0:3]
        nodes[k, 3:12] = R.T.reshape(-1)
        nodes[k, 12:15] = rng.standard_normal(3) * 0.01
        nodes[k, 15] = m[i, 6]
    return np.ascontiguousarray(nodes[np.argsort(nodes[:, 15], kind="stable")])


CONFIGS = {
    # the committed full fixture
    "default": dict(K=(160, 120, 132.0, 132.0, 80.0, 60.0), seed=7, speed=1.0),
    # the sampled fixture (tests/test_gl_golden.py::test_oracle_matches_reference_shaders_live): the ICL-NUIM camera (fx != fy,
    # half-pixel principal point; SURVEY 8d S1) at a quarter and at half of its resolution, and an off-centre camera with another
    # aspect ratio and faster motion
    "icl": dict(K=(160, 120, 481.2 / 4, 480.0 / 4, 319.5 / 4, 239.5 / 4), seed=11, speed=1.0),
    "offcentre": dict(K=(192, 144, 150.0, 155.0, 90.3, 70.7), seed=23, speed=2.0),
    "icl320": dict(K=(320, 240, 481.2 / 2, 480.0 / 2, 319.5 / 2, 239.5 / 2), seed=5, speed=1.5),
}
LIVE_CONFIGS = ("icl", "offcentre", "icl320")


def inputs(config="default"):
    """The inputs of every pass for one configuration, computed with the CPU oracle alone: (dict of arrays, intrinsics)."""
    cfg = CONFIGS[config]
    K = synth.Intrinsics(int(cfg["K"][0]), int(cfg["K"][1]), *[float(x) for x in cfg["K"][2:]])
    frames = list(synth.sequence(8, K, seed=cfg["seed"], noise=True, speed=cfg["speed"]))
    x = {"K": np.array([K.width, K.height, K.fx, K.fy, K.cx, K.cy], np.float64)}
    # ---- frame 0: preprocess + first-frame map
    rgb0, depth0, _ = frames[0]
    x.update(rgb0=rgb0, depth0=depth0, filt0=eo.bilateral(depth0, 3.0))
    # a scene crossing depthCutoff: the two feedback buffers differ in length (SURVEY App. A-29)
    Tb = synth.pose(synth.rot_xyz(0, np.deg2rad(55.0), 0), [-1.6, 0.2, -1.2])
    rgbb, depthb, _, _ = synth.render(Tb, K, noise_seed=77)
    x.update(rgbb=rgbb, depthb=depthb, filtb=eo.bilateral(depthb, 3.0))
    # ---- a map after 4 frames, frame 4 as the measurement
    f = run_oracle(frames, K, 4)
    m, T, tick = f.map(), f.pose, f.tick
    rgb4, depth4, _ = frames[4]
    filt4 = eo.bilateral(depth4, 3.0)
    dm4, dmf4 = eo.metric(depth4, 3.0), eo.metric(filt4, 3.0)
    x.update(map=m, T=T, tick=np.array(tick), rgb4=rgb4, depth4=depth4, filt4=filt4)
    io = eo.predict_indices(m, T, tick, MAXD, BIG, K)  # the chain continues on the oracle's index map (both sides use it)
    x.update(index_in=io[0], vert_conf_in=io[1], color_time_in=io[2], norm_rad_in=io[3])
    fused, new = eo.fuse(m, T, tick, rgb4, dm4, dmf4, *io, MAXD, 0.73, K)
    io2 = eo.predict_indices(fused, T, tick, MAXD, BIG, K)
    x.update(fused_in=fused, new_in=new, index2_in=io2[0], vert_conf2_in=io2[1], color_time2_in=io2[2], norm_rad2_in=io2[3])
    # finite time window + un-cull branch: a map with old time stamps
    mt = fused.copy()
    n = len(mt)
    mt[:, 6] = 1 + np.floor(np.arange(n) * 50.0 / n)
    mt[:, 7] = np.maximum(np.where(np.arange(n) % 2 == 0, 20.0, 58.0), mt[:, 6])
    mt[:, 3] += np.where(np.arange(n) % 3 == 0, 10.0, 0.0).astype(np.float32)
    tick_t, td = 60, 8
    it = eo.predict_indices(mt, T, tick_t, MAXD, td, K)
    x.update(map_t=mt, tick_t=np.array(tick_t), td=np.array(td), index_t_in=it[0], vert_conf_t_in=it[1], color_time_t_in=it[2],
             norm_rad_t_in=it[3])
    # deformation graph inside clean (copy_unstable.vert:132-322)
    x.update(nodes=graph_for(mt), synth_depth_t_in=eo.combined_predict(mt, T, MAXD, 10.0, tick_t, tick_t - td, 65535, K, depth_only=True))
    # ---- model raycast (ACTIVE, INACTIVE, depth) and fill-in
    ms = fused.copy()
    ms[:, 3] += 10.0
    po = eo.combined_predict(ms, T, MAXD, 10.0, tick, tick, BIG, K)
    x.update(map_stable=ms, image_in=po[0], vertex_in=po[1], normal_in=po[2])
    return x, K


def reference(gl, x):
    """What the reference's shaders compute from the inputs x of every pass (a dict of `gl_*` arrays)."""
    T, tick, tick_t, td = x["T"], int(x["tick"]), int(x["tick_t"]), int(x["td"])
    it = (x["index_t_in"], x["vert_conf_t_in"], x["color_time_t_in"], x["norm_rad_t_in"])
    out = {"gl_log": np.array(gl.log())}
    out.update(gl_bilateral=gl.bilateral(x["depth0"], 3.0), gl_metric=gl.metric(x["depth0"], 3.0), gl_metric_filtered=gl.metric(x["filt0"], 3.0))
    dm0, dmf0 = eo.metric(x["depth0"], 3.0), eo.metric(x["filt0"], 3.0)
    raw, fil = gl.feedback_buffer(x["rgb0"], dm0, 1, MAXD), gl.feedback_buffer(x["rgb0"], dmf0, 1, MAXD)
    out.update(gl_feedback_raw=raw, gl_feedback_filt=fil, gl_initial_map=gl.map_initialise(raw, fil))
    rawb = gl.feedback_buffer(x["rgbb"], eo.metric(x["depthb"], 3.0), 1, MAXD)
    filb = gl.feedback_buffer(x["rgbb"], eo.metric(x["filtb"], 3.0), 1, MAXD)
    out.update(gl_boundary_raw_count=np.array(len(rawb)), gl_boundary_filt_count=np.array(len(filb)), gl_boundary_map=gl.map_initialise(rawb, filb))
    m = x["map"]
    ig = gl.predict_indices(m, T, tick, MAXD, BIG)
    out.update(gl_index=ig[0], gl_vert_conf=ig[1], gl_color_time=ig[2], gl_norm_rad=ig[3])
    io = (x["index_in"], x["vert_conf_in"], x["color_time_in"], x["norm_rad_in"])
    fused_gl, new_gl = gl.fuse(m, T, tick, x["rgb4"], eo.metric(x["depth4"], 3.0), eo.metric(x["filt4"], 3.0), *io, MAXD, 0.73)
    out.update(gl_fused=fused_gl, gl_fuse_feedback=new_gl)
    io2 = (x["index2_in"], x["vert_conf2_in"], x["color_time2_in"], x["norm_rad2_in"])
    out.update(gl_cleaned=gl.clean(x["fused_in"], new_gl, T, tick, *io2, 10.0, BIG, MAXD))
    mt = x["map_t"]
    out.update(gl_index_t=gl.predict_indices(mt, T, tick_t, MAXD, td)[0])
    none = np.zeros((0, 12), np.float32)
    out.update(gl_cleaned_t=gl.clean(mt, none, T, tick_t, *it, 10.0, td, MAXD))
    out.update(gl_synth_depth_t=gl.combined_predict(mt, T, MAXD, 10.0, tick_t, tick_t - td, 65535, depth_only=True),
               gl_cleaned_deformed=gl.clean(mt, none, T, tick_t, *it, 10.0, td, MAXD, nodes=x["nodes"], depth=x["synth_depth_t_in"]))
    ms = x["map_stable"]
    pg = gl.combined_predict(ms, T, MAXD, 10.0, tick, tick, BIG)
    out.update(gl_image=pg[0], gl_vertex=pg[1], gl_normal=pg[2], gl_time=pg[3],
               gl_synth_depth=gl.combined_predict(ms, T, MAXD, 10.0, tick, tick, BIG, depth_only=True))
    pin = gl.combined_predict(mt, T, MAXD, 10.0, 0, tick_t - td, td)
    out.update(gl_old_image=pin[0], gl_old_vertex=pin[1], gl_old_normal=pin[2], gl_old_time=pin[3])
    filt4, rgb4 = x["filt4"], x["rgb4"]
    out.update(gl_fill_vertex=gl.fill_vertex(x["vertex_in"], filt4, 0), gl_fill_normal=gl.fill_normal(x["normal_in"], filt4, 0),
               gl_fill_image=gl.fill_image(x["image_in"], rgb4, 0), gl_fill_vertex_pass=gl.fill_vertex(x["vertex_in"], filt4, 1),
               gl_fill_image_pass=gl.fill_image(x["image_in"], rgb4, 1))
    out["gl_error"] = np.array(int(gl.lib.efg_gl_error()))
    return out


def build(config="default"):
    """Inputs and the reference shaders' outputs of every pass for one configuration (a dict of arrays)."""
    from oracle import ef_refgl as rg

    x, K = inputs(config)
    return dict(x, **reference(rg.RefGL(K), x)), K


# ---- the sampled fixture
def PIXELS(h, w):
    return np.arange(0, h * w, PIXEL_STRIDE)


def ROWS(n):
    return np.unique(np.linspace(0, n - 1, min(n, ROW_SAMPLE)).astype(np.int64)) if n else np.zeros(0, np.int64)


def sample_pixels(a, h, w):
    """(h, w[, c]) -> (samples, 1[, c]): an image restricted to PIXELS(), shaped so that per-pixel checks apply unchanged."""
    a = np.asarray(a)
    return a.reshape((h * w,) + a.shape[2:])[PIXELS(h, w)][:, None]


# the shader outputs run_all reads: surfel lists (sampled by ROWS(), their full length kept in `<name>_len`) and images
SURFEL_OUTPUTS = ("gl_initial_map", "gl_boundary_map", "gl_fused", "gl_fuse_feedback", "gl_cleaned", "gl_cleaned_t", "gl_cleaned_deformed")
PIXEL_OUTPUTS = ("gl_bilateral", "gl_metric", "gl_index", "gl_vert_conf", "gl_color_time", "gl_norm_rad", "gl_index_t", "gl_image", "gl_vertex",
                 "gl_normal", "gl_time", "gl_synth_depth", "gl_old_image", "gl_old_vertex", "gl_old_normal", "gl_old_time", "gl_fill_vertex",
                 "gl_fill_normal", "gl_fill_image", "gl_fill_vertex_pass", "gl_fill_image_pass")


def sampled(G, K):
    """The shader outputs run_all reads, sampled. gl_fuse_feedback keeps only its new surfels (w = -2): all that run_all takes
    from it once check_fixture has seen the whole array."""
    out = {k: G[k] for k in ("gl_log", "gl_error", "gl_boundary_raw_count", "gl_boundary_filt_count")}
    fb = G["gl_fuse_feedback"]
    for k in SURFEL_OUTPUTS:
        a = fb[fb[:, 7] == -2] if k == "gl_fuse_feedback" else G[k]
        out[k], out[f"{k}_len"] = a[ROWS(len(a))], np.array(len(a))
    for k in PIXEL_OUTPUTS:
        out[k] = sample_pixels(G[k], K.height, K.width)
    return out


def main():
    from oracle import ef_refgl as rg

    if not rg.in_gl_process():
        if not rg.available():
            raise SystemExit("oracle/_ref/gl is not built (make -C oracle refgl) or Mesa / the reference tree is absent")
        if sys.argv[1:] == ["--live"]:
            # one GL process per configuration (a process holds one GL context), merged into one file
            import tempfile

            z = {}
            with tempfile.TemporaryDirectory() as tmp:
                for config in LIVE_CONFIGS:
                    part = os.path.join(tmp, config + ".npz")
                    rg.run_script(os.path.abspath(__file__), "--live-one", config, part)
                    z.update(np.load(part))
            np.savez_compressed(LIVE_PATH, **z)
            print("wrote", LIVE_PATH, os.path.getsize(LIVE_PATH) // 1024, "KiB")
            return
        rg.run_script(os.path.abspath(__file__), *sys.argv[1:])
        return
    import test_gl_golden as tg

    if len(sys.argv) > 2 and sys.argv[1] == "--check":
        # the oracle compared with what the shaders just produced, with the same pass-by-pass checks the fixture test applies
        out, K = build(sys.argv[2])
        assert int(out["gl_error"]) == 0 and "llvmpipe" in str(out["gl_log"])
        tg.check_fixture(out)
        tg.run_all(tg.Oracle(K), out, K, False)
        print("LIVE OK", sys.argv[2])
        return
    if len(sys.argv) > 3 and sys.argv[1] == "--live-one":
        config, path = sys.argv[2], sys.argv[3]
        x, K = inputs(config)
        G = dict(x, **reference(rg.RefGL(K), x))
        assert int(G["gl_error"]) == 0 and "llvmpipe" in str(G["gl_log"])
        tg.check_fixture(G)
        z = {f"{config}/inputs_sha256": np.array(digest(x))}
        z.update({f"{config}/{k}": v for k, v in sampled(G, K).items()})
        np.savez(path, **z)
        return
    out, _ = build("default")
    path = os.path.join(ROOT, "tests", "golden", "ref_mapping_160x120.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB; gl error", int(out["gl_error"]))
    print(out["gl_log"])


if __name__ == "__main__":
    main()
