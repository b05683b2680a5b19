"""The mapping half against the REFERENCE'S OWN GLSL SHADERS: tests/golden/ref_mapping_160x120.npz holds the outputs of the
reference's Core/Shaders/*.{vert,geom,frag} (unmodified) executed on Mesa llvmpipe by oracle/gl/ref_gl_harness.cpp (generator:
tests/golden/make_gl_golden.py). Every pass of the GL half is compared on the inputs stored with it:

  * CPU (`not gpu`): oracle/efo_map.cpp, the restatement that all other mapping tests use as their checker -- this is what pins it;
  * `-m gpu`: libefusion.so through the C ABI.

Tolerances: integer / index / byte outputs must be identical except for a stated fraction of pixels where a value sits on a
rounding boundary (sub-pixel snapping of a window coordinate at x.5/256, exp() in the bilateral weight, pow(r, 2) at a disc edge:
Mesa evaluates transcendental functions with its own polynomials); float outputs 1e-5 absolute (depths are metres)."""
import os
import sys

import numpy as np
import pytest

from util import assert_same, digest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MAXD, BIG = 20.0, 2 ** 30
COLS = [0, 1, 2, 4, 5, 6, 7, 8, 9, 10, 11]  # everything but the confidence (exp())
SAMPLED = False  # True while run_all checks the sampled live fixture (see few())


@pytest.fixture(scope="module")
def G():
    z = np.load(os.path.join(ROOT, "tests", "golden", "ref_mapping_160x120.npz"))
    assert int(z["gl_error"]) == 0 and "llvmpipe" in str(z["gl_log"])
    check_fixture(z)
    return z


@pytest.fixture(scope="module")
def K(G):
    from elasticfusion_b200 import synth

    w, h, fx, fy, cx, cy = G["K"]
    return synth.Intrinsics(int(w), int(h), float(fx), float(fy), float(cx), float(cy))


def differ(a, b, tol=0.0):
    """Per pixel (per surfel for (n, 12) lists): does a differ from b by more than tol (NaN == NaN)?"""
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, (a.shape, b.shape)
    if a.dtype.kind == "f":
        both_nan = np.isnan(a) & np.isnan(b)
        d = np.where(both_nan, 0.0, np.abs(a.astype(np.float64) - b.astype(np.float64)))
        bad = ~(d <= tol)
    else:
        bad = a != b
    if bad.ndim > 2:
        bad = bad.reshape(bad.shape[0], bad.shape[1], -1).any(axis=2)
    elif bad.ndim == 2 and a.shape[1] == 12:
        bad = bad.any(axis=1)
    return bad


def frac_differ(a, b, tol=0.0):
    return float(differ(a, b, tol).mean())


def few(bad, limit):
    """At most a fraction `limit` of the elements are bad. On a sample (the live fixture) a few boundary cases more or less
    than the whole image holds can fall into it: the count may then exceed limit x n by three binomial standard deviations
    and one element."""
    k, allowed = int(np.sum(bad)), limit * np.size(bad)
    if SAMPLED:
        allowed += 3.0 * np.sqrt(allowed) + 1.0
    return k <= allowed


def mad(a, b):
    """max |a - b| with NaN == NaN (the reference's maps carry NaN normals at depth edges); a one-sided NaN counts as inf."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    d = np.abs(a - b)
    d[np.isnan(a) & np.isnan(b)] = 0.0
    d[np.isnan(d)] = np.inf
    return float(d.max()) if d.size else 0.0


def check_surfels(got, ref, what, tol=1e-5, frac=0.0):
    assert len(got) == len(ref), (what, len(got), len(ref))
    assert frac_differ(got[:, COLS], ref[:, COLS], tol) <= frac, (what, frac_differ(got[:, COLS], ref[:, COLS], tol))
    ok = ~np.isnan(ref[:, 3])
    assert np.abs(got[ok, 3] - ref[ok, 3]).max() <= 1e-5 * max(1.0, np.abs(ref[ok, 3]).max()), what


class Oracle:
    """oracle/efo_map.cpp behind the same call names the product side offers below."""

    def __init__(self, K):
        from oracle import ef_oracle as eo

        self.eo, self.K = eo, K

    def bilateral(self, depth):
        return self.eo.bilateral(depth, 3.0)

    def metric(self, depth):
        return self.eo.metric(depth, 3.0)

    def first_frame(self, rgb, depth, filt):
        eo = self.eo
        raw = eo.feedback_buffer(rgb, eo.metric(depth, 3.0), self.K, 1, MAXD)
        fil = eo.feedback_buffer(rgb, eo.metric(filt, 3.0), self.K, 1, MAXD)
        return eo.map_initialise(raw, fil), len(raw), len(fil)

    def predict_indices(self, m, T, tick, td):
        return self.eo.predict_indices(m, T, tick, MAXD, td, self.K)

    def fuse(self, m, T, tick, rgb, depth, filt, idx, w):
        eo = self.eo
        return eo.fuse(m, T, tick, rgb, eo.metric(depth, 3.0), eo.metric(filt, 3.0), *idx, MAXD, w, self.K)

    def clean(self, m, new, T, tick, idx, td, nodes=None, depth=None):
        if nodes is None:
            return self.eo.clean(m, new, T, tick, *idx, 10.0, td, MAXD, self.K)
        return self.eo.clean_deform(m, new, T, tick, idx[0], idx[1], idx[2], 10.0, td, MAXD, self.K, nodes, depth)

    def raycast(self, m, T, time, max_time, td, depth_only=False):
        return self.eo.combined_predict(m, T, MAXD, 10.0, time, max_time, td, self.K, depth_only=depth_only)

    def fill(self, vertex, normal, image, filt, rgb, passthrough):
        eo = self.eo
        return eo.fill_vertex(vertex, filt, passthrough, self.K), eo.fill_normal(normal, filt, passthrough, self.K), eo.fill_image(image, rgb, passthrough)

    def close(self):
        pass


class Product:
    """libefusion.so through the C ABI (stage entry points)."""

    def __init__(self, K):
        from elasticfusion_b200 import capi

        self.K = K
        self.ctx = capi.Context(capi.default_config(K.width, K.height, K.fx, K.fy, K.cx, K.cy, capacity=200000, time_delta=BIG))

    def close(self):
        self.ctx.close()

    def _pre(self, depth):
        c = self.ctx
        c.upload("DEPTH_RAW", depth)
        c.preprocess_depth(c.buffer_ptr("DEPTH_RAW")[0], 3.0, c.buffer_ptr("DEPTH_FILTERED")[0], c.buffer_ptr("DEPTH_METRIC")[0],
                           c.buffer_ptr("DEPTH_METRIC_FILTERED")[0])

    def bilateral(self, depth):
        self._pre(depth)
        return self.ctx.download("DEPTH_FILTERED")

    def metric(self, depth):
        self._pre(depth)
        return self.ctx.download("DEPTH_METRIC")

    def _inputs(self, rgb, depth, filt):
        from oracle import ef_oracle as eo  # (the checker's metric conversion is bit-exact with the product's, asserted above)

        c = self.ctx
        c.upload("RGB", rgb)
        c.upload("DEPTH_RAW", depth)
        c.upload("DEPTH_FILTERED", filt)
        c.upload("DEPTH_METRIC", eo.metric(depth, 3.0))
        c.upload("DEPTH_METRIC_FILTERED", eo.metric(filt, 3.0))

    def first_frame(self, rgb, depth, filt):
        self._inputs(rgb, depth, filt)
        self.ctx.map_initialise()
        return self.ctx.map_download(), None, None

    def _upload_index(self, idx):
        for name, a in zip(("INDEX", "VERT_CONF", "COLOR_TIME", "NORM_RAD"), idx):
            self.ctx.upload(name, a)

    def predict_indices(self, m, T, tick, td):
        c = self.ctx
        c.map_upload(m)
        c.map_predict_indices(T, tick, MAXD, td)
        return tuple(c.download(n) for n in ("INDEX", "VERT_CONF", "COLOR_TIME", "NORM_RAD"))

    def fuse(self, m, T, tick, rgb, depth, filt, idx, w):
        c = self.ctx
        self._inputs(rgb, depth, filt)
        c.map_upload(m)
        self._upload_index(idx)
        c.map_fuse(T, tick, MAXD, w)
        return c.map_download(), c.map_download_new()

    def clean(self, m, new, T, tick, idx, td, nodes=None, depth=None):
        c = self.ctx
        c.map_upload(m)
        assert len(new) == 0 or self._new_ready, "new surfels come from the preceding fuse on this context"
        self._upload_index(idx)
        if nodes is None:
            c.map_clean(T, tick, 10.0, td, MAXD)
        else:
            c.upload("SYNTH_DEPTH", depth)
            c.map_clean_deform(T, tick, 10.0, td, MAXD, nodes)
        return c.map_download()

    _new_ready = False

    def raycast(self, m, T, time, max_time, td, depth_only=False, mode=0):
        c = self.ctx
        c.map_upload(m)
        if depth_only:
            c.map_raycast(T, MAXD, 10.0, time, max_time, td, 2)
            return c.download("SYNTH_DEPTH")
        c.map_raycast(T, MAXD, 10.0, time, max_time, td, mode)
        names = ("IMAGE", "VERTEX", "NORMAL", "TIME") if mode == 0 else ("OLD_IMAGE", "OLD_VERTEX", "OLD_NORMAL", "OLD_TIME")
        return tuple(c.download(n) for n in names)

    def fill(self, vertex, normal, image, filt, rgb, passthrough):
        c = self.ctx
        c.upload("VERTEX", vertex)
        c.upload("NORMAL", normal)
        c.upload("IMAGE", image)
        c.upload("DEPTH_FILTERED", filt)
        c.upload("RGB", rgb)
        c.map_fill_in(bool(passthrough), bool(passthrough))
        return c.download("FILL_VERTEX"), c.download("FILL_NORMAL"), c.download("FILL_IMAGE")


def check_fixture(G):
    """The cases the fixture must exercise, read from the reference's outputs in full."""
    assert (np.abs(G["gl_fused"][:, :3] - G["map"][:, :3]).max(axis=1) > 0).sum() > 1000
    fb = G["gl_fuse_feedback"]  # everything the data pass fed back: matched measurements (w = -1) and new surfels (w = -2)
    assert (fb[:, 7] == -2).sum() > 0 and (fb[:, 7] == -1).sum() > 1000
    mt = G["map_t"]
    stale = (int(G["tick_t"]) - mt[:, 7] > 20) & (mt[:, 3] < 10.0)
    assert stale.sum() > 1000 and len(G["gl_cleaned_t"]) == len(mt)  # copy_unstable.vert:126-128 un-culls what left the time window


class Sampled:
    """An oracle whose outputs are cut to the samples of the live fixture (make_gl_golden.sample_pixels / ROWS). Surfel lists come
    in run_all's call order; each one's full length is checked against the reference's before it is cut."""

    def __init__(self, S, G, K):
        import make_gl_golden as mg

        self.S, self.G, self.K, self.mg = S, G, K, mg
        self.lists = iter(mg.SURFEL_OUTPUTS)

    def _rows(self, a):
        name = next(self.lists)
        assert len(a) == int(self.G[name + "_len"]), (name, len(a), int(self.G[name + "_len"]))
        return a[self.mg.ROWS(len(a))]

    def _px(self, a):
        return self.mg.sample_pixels(a, self.K.height, self.K.width)

    def bilateral(self, depth):
        return self._px(self.S.bilateral(depth))

    def metric(self, depth):
        return self._px(self.S.metric(depth))

    def first_frame(self, rgb, depth, filt):
        m, n_raw, n_fil = self.S.first_frame(rgb, depth, filt)
        return self._rows(m), n_raw, n_fil

    def predict_indices(self, m, T, tick, td):
        return tuple(self._px(a) for a in self.S.predict_indices(m, T, tick, td))

    def fuse(self, *args):
        fused, new = self.S.fuse(*args)
        return self._rows(fused), self._rows(new)

    def clean(self, *args, **kw):
        return self._rows(self.S.clean(*args, **kw))

    def raycast(self, *args, **kw):
        out = self.S.raycast(*args, **kw)
        return self._px(out) if isinstance(out, np.ndarray) else tuple(self._px(a) for a in out)

    def fill(self, *args):
        return tuple(self._px(a) for a in self.S.fill(*args))


def run_all(S, G, K, is_product):
    T, tick = G["T"], int(G["tick"])
    # ---- depth_bilateral.frag / depth_metric.frag
    d = np.abs(S.bilateral(G["depth0"]).astype(np.int32) - G["gl_bilateral"].astype(np.int32))
    assert d.max() <= 1 and few(d > 0, 2e-3), (d.max(), (d > 0).mean())  # exp() of the range weight
    assert np.array_equal(S.metric(G["depth0"]) == 0, G["gl_metric"] == 0)
    assert np.abs(S.metric(G["depth0"]) - G["gl_metric"]).max() <= 2.4e-7  # one ulp: value / 1000.0f
    # ---- vertex_feedback.vert/.geom + init_unstable.vert
    m0, n_raw, n_fil = S.first_frame(G["rgb0"], G["depth0"], G["filt0"])
    check_surfels(m0, G["gl_initial_map"], "first-frame map", tol=1e-6)
    assert np.array_equal(m0[:, :3], G["gl_initial_map"][:, :3]) and np.array_equal(m0[:, 4:8], G["gl_initial_map"][:, 4:8])
    mb, nb_raw, nb_fil = S.first_frame(G["rgbb"], G["depthb"], G["filtb"])
    assert int(G["gl_boundary_raw_count"]) != int(G["gl_boundary_filt_count"])  # the App. A-29 case is exercised
    if n_raw is not None:
        assert (nb_raw, nb_fil) == (int(G["gl_boundary_raw_count"]), int(G["gl_boundary_filt_count"]))
    check_surfels(mb, G["gl_boundary_map"], "first-frame map across depthCutoff", tol=1e-6)
    # ---- index_map.vert/.frag (incl. the time-window cull)
    idx = S.predict_indices(G["map"], T, tick, BIG)
    assert few(differ(idx[0], G["gl_index"]), 5e-4)  # a window coordinate within float rounding of a snapping boundary
    same = idx[0] == G["gl_index"]
    for a, name in zip(idx[1:], ("gl_vert_conf", "gl_color_time", "gl_norm_rad")):
        assert mad(a[same], G[name][same]) <= 1e-6, name
    assert (G["gl_index"] > 0).mean() > 0.5
    idx_t = S.predict_indices(G["map_t"], T, int(G["tick_t"]), int(G["td"]))
    assert few(differ(idx_t[0], G["gl_index_t"]), 5e-4) and 0.1 < (G["gl_index_t"] > 0).mean() < 0.9
    # ---- data.vert/.geom/.frag + update.vert
    idx_in = (G["index_in"], G["vert_conf_in"], G["color_time_in"], G["norm_rad_in"])
    fused, new = S.fuse(G["map"], T, tick, G["rgb4"], G["depth4"], G["filt4"], idx_in, 0.73)
    check_surfels(fused, G["gl_fused"], "fused map", tol=1e-5)
    fb = G["gl_fuse_feedback"]
    check_surfels(new, fb[fb[:, 7] == -2], "new unstable surfels", tol=1e-5)
    # ---- copy_unstable.vert/.geom
    idx2 = (G["index2_in"], G["vert_conf2_in"], G["color_time2_in"], G["norm_rad2_in"])
    if is_product:
        S._new_ready = True  # the product's new-surfel buffer holds what its fuse just emitted
        S.ctx.map_upload(G["fused_in"])
    cleaned = S.clean(G["fused_in"], G["new_in"], T, tick, idx2, BIG)
    check_surfels(cleaned, G["gl_cleaned"], "map after clean", tol=1e-6)
    idx_tin = (G["index_t_in"], G["vert_conf_t_in"], G["color_time_t_in"], G["norm_rad_t_in"])
    none = np.zeros((0, 12), np.float32)
    if is_product:
        S._new_ready = False
        S.ctx.map_upload(G["map_t"][:1])
        S.ctx.map_clean(T, int(G["tick_t"]), 10.0, int(G["td"]), MAXD)  # (drains the new-surfel buffer of the fuse above)
    cleaned_t = S.clean(G["map_t"], none, T, int(G["tick_t"]), idx_tin, int(G["td"]))
    check_surfels(cleaned_t, G["gl_cleaned_t"], "map after clean, finite time window", tol=1e-6)
    # ---- copy_unstable.vert with a deformation graph (lines 132-322)
    deformed = S.clean(G["map_t"], none, T, int(G["tick_t"]), idx_tin, int(G["td"]), nodes=G["nodes"], depth=G["synth_depth_t_in"])
    ref = G["gl_cleaned_deformed"]
    assert len(deformed) == len(ref) and np.nanmax(np.abs(ref[:, :3] - G["gl_cleaned_t"][:, :3])) > 1e-3
    assert np.array_equal(np.isnan(deformed), np.isnan(ref))
    ok = ~np.isnan(ref).any(axis=1)
    assert np.abs(deformed[ok][:, [0, 1, 2, 8, 9, 10]] - ref[ok][:, [0, 1, 2, 8, 9, 10]]).max() <= 2e-5
    assert few(deformed[ok, 7] != ref[ok, 7], 1e-3)  # lastTime refresh: a depth comparison at a 10 cm margin
    # ---- splat.vert + combo_splat.frag / depth_splat.frag: ACTIVE, INACTIVE, depth only
    for m, time, max_time, td, names, mode in ((G["map_stable"], tick, tick, BIG, ("gl_image", "gl_vertex", "gl_normal", "gl_time"), 0),
                                               (G["map_t"], 0, int(G["tick_t"]) - int(G["td"]), int(G["td"]),
                                                ("gl_old_image", "gl_old_vertex", "gl_old_normal", "gl_old_time"), 1)):
        out = S.raycast(m, T, time, max_time, td, mode=mode) if is_product else S.raycast(m, T, time, max_time, td)
        assert few(differ(out[0], G[names[0]]), 5e-4) and few(differ(out[3], G[names[3]]), 5e-4), names  # pow(r, 2) at a disc edge
        same = (out[3] == G[names[3]]) & (out[0] == G[names[0]]).all(axis=2)
        # (1e-5 m but for a handful of fragments where the ray grazes its disc and the intersection's division amplifies the last
        # bits: 3 of 307 k values reach 1.9e-5 at 320x240)
        assert mad(out[1][same], G[names[1]][same]) <= 5e-5 and mad(out[2][same], G[names[2]][same]) <= 1e-5
        assert few(differ(out[1][same], G[names[1]][same], 1e-5), 1e-4)
        assert (G[names[1]][..., 2] > 0).mean() > 0.2
    sd = S.raycast(G["map_stable"], T, tick, tick, BIG, depth_only=True)
    assert few(differ(sd, G["gl_synth_depth"], 1e-5), 5e-4)
    # ---- fill_vertex / fill_normal / fill_rgb
    for p, (kv, kn, ki) in ((0, ("gl_fill_vertex", "gl_fill_normal", "gl_fill_image")), (1, ("gl_fill_vertex_pass", None, "gl_fill_image_pass"))):
        fv, fn, fi = S.fill(G["vertex_in"], G["normal_in"], G["image_in"], G["filt4"], G["rgb4"], p)
        assert frac_differ(fv, G[kv], 1e-6) == 0
        if kn:
            assert few(differ(fn, G[kn], 1e-4), 1e-3)  # normalize(): rsqrt polynomial
        assert_same(fi, G[ki], ki)


def test_oracle_matches_reference_shaders(G, K):
    """oracle/efo_map.cpp == the reference's GLSL on Mesa, pass by pass: the pin of the GL half of the oracle."""
    S = Oracle(K)
    run_all(S, G, K, False)


@pytest.mark.parametrize("config", ["icl", "offcentre", "icl320"])
def test_oracle_matches_reference_shaders_live(config, monkeypatch):
    """The same pin in configurations the full fixture does not hold -- the ICL-NUIM camera (fx != fy, half-pixel principal
    point) at two resolutions and an off-centre camera with another aspect ratio and faster motion. The oracle regenerates the
    inputs of every pass; tests/golden/ref_mapping_live.npz holds their digest and a fixed sample of what the reference's shaders
    computed from them (make_gl_golden.py --live), and the same pass-by-pass checks run on that sample."""
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import make_gl_golden as mg

    z = np.load(os.path.join(ROOT, "tests", "golden", "ref_mapping_live.npz"))
    x, K = mg.inputs(config)
    assert digest(x) == str(z[f"{config}/inputs_sha256"]), "the inputs changed: regenerate with make_gl_golden.py --live"
    G = dict(x, **{k.split("/", 1)[1]: z[k] for k in z.files if k.startswith(config + "/")})
    assert int(G["gl_error"]) == 0 and "llvmpipe" in str(G["gl_log"])
    monkeypatch.setattr(sys.modules[__name__], "SAMPLED", True)
    run_all(Sampled(Oracle(K), G, K), G, K, False)


@pytest.mark.gpu
def test_product_matches_reference_shaders(G, K):
    """libefusion.so == the reference's GLSL on Mesa, pass by pass, through the C ABI."""
    S = Product(K)
    try:
        run_all(S, G, K, True)
    finally:
        S.close()
