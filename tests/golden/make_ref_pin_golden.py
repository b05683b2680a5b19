"""Generates tests/golden/ref_pin_640x480.npz ON A GPU from the REFERENCE's own CUDA tracking kernels (oracle/_ref/libef_ref.so:
Core/Cuda/reduce.cu + cudafuncs.cu compiled unmodified from the reference tree by `make -C oracle ref`).

    python tests/golden/make_ref_pin_golden.py [OUT.npz]

The inputs are those of tests/test_gpu_ref_pin.py (the 640x480 sequence of tests/conftest.py through three frames of the CPU
oracle); they are not stored, only their digest, so the test can tell a changed input from a changed result. What the reference
computed is stored so that the file stays small: the NaN masks of every pyramid map in full, the map values at a fixed seeded
sample of pixels with their full sums and largest magnitude, sha256 digests of the integer depth pyramid, and the ICP steps and
the whole tracking run (6x6 systems, residuals, per-iteration trace, final pose) in full."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from elasticfusion_b200 import synth  # noqa: E402
from oracle import ef_ref  # noqa: E402
from util import digest, pose_inputs, tracking_inputs  # noqa: E402

LEVELS = (0, 1, 2)
SAMPLE = {0: 4096, 1: 2048, 2: 1024}  # pixels per level
MAPS = ("vmap_curr", "nmap_curr", "vmap_g_prev", "nmap_g_prev")
DEPTHS = ("lastDepth", "nextDepth")
IMAGES = ("lastImage", "nextImage", "lastNextImage")


def main(out):
    if not ef_ref.available():
        raise SystemExit("oracle/_ref/libef_ref.so is not built (make -C oracle ref) or no GPU is visible")
    K = synth.K_DEFAULT
    frames = list(synth.sequence(8, K, seed=42, noise=True))  # the `frames` fixture of tests/conftest.py
    x = tracking_inputs(frames, K)
    ref = ef_ref.RefOdometry(K)
    ref.init_first_rgb(x["prev_rgba"])
    ref.init_icp_model(x["vtx"], x["nrm"], x["T"])
    ref.init_rgb_model(x["img"])
    ref.init_icp_depth(x["filt"], 20.0)
    ref.init_rgb(x["rgba"])
    g = {"inputs_sha256": np.array(digest(x))}
    rng = np.random.default_rng(20261017)
    for lv in LEVELS:
        r, c = K.height >> lv, K.width >> lv
        idx = np.sort(rng.choice(r * c, SAMPLE[lv], replace=False)).astype(np.int32)
        g[f"idx{lv}"] = idx
        g[f"depth_tmp{lv}_sha256"] = np.array(digest({"a": ref.buffer("depth_tmp", lv)}))
        for n in MAPS:
            planes = ref.buffer(n, lv).reshape(3, r * c)
            valid = ~np.isnan(planes[0])
            g[f"{n}{lv}_nan"] = np.packbits(~valid)
            g[f"{n}{lv}_s"] = planes[:, idx]
            v = planes[:, valid].astype(np.float64)
            g[f"{n}{lv}_stats"] = np.array([v.sum(), np.abs(v).sum(), np.abs(v).max()])
        for n in DEPTHS:
            a = ref.buffer(n, lv).reshape(-1)
            g[f"{n}{lv}_nan"] = np.packbits(np.isnan(a))
            g[f"{n}{lv}_s"] = a[idx]
        for n in IMAGES:
            g[f"{n}{lv}_s"] = ref.buffer(n, lv).reshape(-1)[idx]
    Rc, tc, Rpi, tp = pose_inputs(x["T"])
    for lv in LEVELS:
        A, b, res = ref.icp_step(lv, Rc, tc, Rpi, tp)
        g[f"icp_A{lv}"], g[f"icp_b{lv}"], g[f"icp_r{lv}"] = A, b, res
    Tr, tr = ref.track(x["T"])
    g["track_T"] = Tr
    g["track_trace"] = tr.view(np.uint8)
    np.savez_compressed(out, **g)
    print("wrote", out, os.path.getsize(out), "bytes;", len(tr), "trace records; inputs", g["inputs_sha256"])


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden", "ref_pin_640x480.npz"))
