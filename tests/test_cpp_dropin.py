"""The source-level drop-in: the reference README's Core-API program (tests/cpp/core_api_example.cpp, written against
`#include <ElasticFusion.h>`) must compile against include/efusion/ + libefusion.so, and on a GPU produce the same pose
and surfel count as the C ABI driven from Python."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "core_api_example.cpp")
CUDA_LIB = "/usr/local/cuda/lib64"


def _compile(out, extra=()):
    cmd = ["/usr/bin/g++", "-std=c++17", "-O1", "-Wall", "-Werror", f"-I{ROOT}/include/efusion", f"-I{ROOT}/include", *extra, SRC, "-o", out,
           f"-L{ROOT}/elasticfusion_b200", "-lefusion", f"-Wl,-rpath,{ROOT}/elasticfusion_b200", f"-L{CUDA_LIB}", "-lcudart"]
    subprocess.check_call(cmd)


def test_core_api_example_compiles(tmp_path):
    _compile(str(tmp_path / "example"))


def test_core_api_example_compiles_with_reference_sophus(tmp_path):
    """With the reference's vendored Sophus + Eigen on the include path the pose type is Sophus::SE3d, as in the reference. The
    reference tree is the one oracle/Makefile builds from (REF)."""
    ref = subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "print-ref"], capture_output=True, text=True).stdout.strip()
    third = os.path.join(ref, "third-party")
    if not ref or not os.path.isdir(os.path.join(third, "Sophus")):
        pytest.skip("reference tree not present")
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-fsyntax-only", "-DEIGEN_MAX_ALIGN_BYTES=0", f"-I{third}/Sophus", f"-I{third}/Eigen",
                           f"-I{ROOT}/include/efusion", f"-I{ROOT}/include", SRC])


@pytest.mark.gpu
def test_core_api_example_runs_and_matches_c_abi(tmp_path, small_K, small_frames):
    from elasticfusion_b200 import capi, synth

    exe = str(tmp_path / "example")
    _compile(exe)
    klg = str(tmp_path / "seq.klg")
    synth.write_klg(klg, [(f[0], f[1]) for f in small_frames])
    K = small_K
    out = subprocess.check_output([exe, klg, str(K.width), str(K.height), str(K.fx), str(K.fy), str(K.cx), str(K.cy)], text=True)
    # the same program handing processFrame the next frame as well (look-ahead) must print exactly the same result
    out_la = subprocess.check_output([exe, klg, str(K.width), str(K.height), str(K.fx), str(K.fy), str(K.cx), str(K.cy), "lookahead"], text=True)
    assert out_la == out
    pose = np.array([float(x) for x in out.split("POSE")[1].split("\n")[0].split()]).reshape(4, 4)
    count = int(out.split("COUNT")[1].split()[0])
    tick = int(out.split("TICK")[1].split()[0])
    ctx = capi.Context(capi.default_config(K.width, K.height, K.fx, K.fy, K.cx, K.cy, capacity=500000, time_delta=2147483647 // 2))
    try:
        for i, (rgb, d, _) in enumerate(small_frames):
            ctx.process_frame(rgb, d, i * 33333)
        assert np.abs(ctx.get_pose() - pose).max() < 1e-8
        assert ctx.map_count() == count and ctx.get_tick() == tick == len(small_frames) + 1
        surfels = ctx.map_download()
    finally:
        ctx.close()
    assert os.path.exists("/tmp/ef_b200_example.freiburg")
    lines = open("/tmp/ef_b200_example.freiburg").read().strip().split("\n")
    assert len(lines) == len(small_frames) and len(lines[0].split()) == 8

    # savePly (Core/ElasticFusion.cpp:684-781): ASCII header, then per surfel with confidence > threshold: xyz float32 LE,
    # r g b bytes of the 24-bit colour, NEGATED normal and the radius as float32
    raw = open("/tmp/ef_b200_example.ply", "rb").read()
    head, _, body = raw.partition(b"end_header\n")
    lines = head.decode().split("\n")
    assert lines[0] == "ply" and lines[1] == "format binary_little_endian 1.0"
    props = [l for l in lines if l.startswith("property")]
    assert props == ["property float x", "property float y", "property float z", "property uchar red", "property uchar green", "property uchar blue",
                     "property float nx", "property float ny", "property float nz", "property float radius"]
    keep = surfels[surfels[:, 3] > np.float32(0.9)]
    n = int([l for l in lines if l.startswith("element vertex")][0].split()[-1])
    assert n == len(keep) and 0 < n < len(surfels) and len(body) == n * 31
    rec = np.frombuffer(body, np.dtype([("p", "<f4", 3), ("c", "u1", 3), ("n", "<f4", 4)]))
    assert np.array_equal(rec["p"], keep[:, 0:3])
    col = keep[:, 4].astype(np.int64)
    assert np.array_equal(rec["c"], np.stack([(col >> 16) & 255, (col >> 8) & 255, col & 255], 1).astype(np.uint8))
    nz = ~np.isnan(keep[:, 8:11]).any(axis=1)
    assert np.array_equal(rec["n"][nz, :3], -keep[nz, 8:11]) and np.array_equal(rec["n"][:, 3], keep[:, 11])


@pytest.mark.gpu
def test_headless_cli_matches_c_abi(tmp_path, small_K, small_frames):
    """tools/ElasticFusionHeadless (the reference application's flags, MainController.cpp:32-104, without GUI): `-l log -cal file -o`
    over a zlib + raw .klg must leave a .freiburg whose last pose equals the C ABI run's. hasMore() drops the last frame of a log
    (RawLogReader.cpp:139-141), so N-1 frames are processed."""
    import zlib, struct
    from elasticfusion_b200 import capi

    exe = os.path.join(ROOT, "tools", "ElasticFusionHeadless")
    if not os.path.exists(exe):
        subprocess.check_call(["bash", os.path.join(ROOT, "build.sh")])
    K = small_K
    klg = str(tmp_path / "cli.klg")
    with open(klg, "wb") as f:
        f.write(struct.pack("<i", len(small_frames)))
        for i, (rgb, depth, _) in enumerate(small_frames):
            db = zlib.compress(depth.astype("<u2").tobytes()) if i % 2 else depth.astype("<u2").tobytes()
            ib = rgb.tobytes()
            f.write(struct.pack("<qii", i * 33333, len(db), len(ib)))
            f.write(db)
            f.write(ib)
    cal = str(tmp_path / "cal.txt")
    open(cal, "w").write(f"{K.fx} {K.fy} {K.cx} {K.cy}\n")
    outs = []
    for extra in ([], ["-nola"]):
        out = subprocess.check_output([exe, "-l", klg, "-cal", cal, "-w", str(K.width), "-h", str(K.height), "-o", "-cap", "500000", "-ply", "-v"] + extra, text=True)
        outs.append([l for l in out.split("\n") if l.startswith("frame ")])
        assert f"{len(small_frames) - 1} frames" in out
    assert [l.rsplit(" ", 2)[0] for l in outs[0]] == [l.rsplit(" ", 2)[0] for l in outs[1]]  # look-ahead changes nothing but the time
    lines = open(klg + ".freiburg").read().strip().split("\n")
    assert len(lines) == len(small_frames) - 1
    ctx = capi.Context(capi.default_config(K.width, K.height, K.fx, K.fy, K.cx, K.cy, capacity=500000, time_delta=2147483647 // 2))
    try:
        for i, (rgb, d, _) in enumerate(small_frames[:-1]):
            ctx.process_frame(rgb, d, i * 33333)
        T = ctx.get_pose()
    finally:
        ctx.close()
    last = [float(x) for x in lines[-1].split()]
    assert abs(last[0] - (len(small_frames) - 2) * 33333 / 1e6) < 1e-6
    assert np.abs(np.array(last[1:4]) - T[:3, 3]).max() < 1e-5
    assert os.path.getsize(klg + ".ply") > 100


@pytest.mark.gpu
def test_ferns_keyframes_and_relocalisation_candidate(tmp_path, K):
    """include/efusion/Ferns.h (Core/Ferns.h:36-166, Ferns.cpp:22-420): frames are encoded at W/8 x H/8 and stored when dissimilar
    enough; findFrame on a revisited view proposes a stored frame and its 80x60 ICP-only registration (third RGBDOdometry
    instance of the reference) recovers the camera pose; 50-sample surface constraints come back."""
    from elasticfusion_b200 import synth

    exe = str(tmp_path / "ferns_check")
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O1", "-Wall", "-Werror", f"-I{ROOT}/include/efusion", f"-I{ROOT}/include",
                           os.path.join(ROOT, "tests", "cpp", "ferns_check.cpp"), "-o", exe, f"-L{ROOT}/elasticfusion_b200", "-lefusion",
                           f"-Wl,-rpath,{ROOT}/elasticfusion_b200", f"-L{CUDA_LIB}", "-lcudart", "-lz"])
    # A floor corner (three planes inside the depth cut-off: the ICP-only registration is constrained in all six degrees of
    # freedom; over the default views it slides along the walls, on the oracle as well), walked out, half way back and out
    # again: the last processed frame revisits view 14, next to a key frame stored on the way out.
    out_leg = list(synth.corner_sequence(16, K, seed=17, noise=True, speed=3.0))
    order = list(range(16)) + list(range(14, 8, -1)) + list(range(10, 16)) + [15, 14, 14]
    frames = [out_leg[i] for i in order]
    assert len(frames) == 31
    klg = str(tmp_path / "ferns.klg")
    synth.write_klg(klg, [(f[0], f[1]) for f in frames])
    run = subprocess.run([exe, klg, str(K.width), str(K.height), str(K.fx), str(K.fy), str(K.cx), str(K.cy), "400", "2"], text=True, capture_output=True, check=True)
    out = run.stdout
    print(run.stderr)
    kv = dict(zip(out.split()[0::2], out.split()[1::2]))
    assert int(kv["FRAMES"]) == 30 and int(kv["STORED"]) >= 2 and int(kv["STORED"]) == int(kv["ADDED"])
    assert int(kv["CLOSEST"]) >= 0, out + run.stderr
    assert float(kv["ICPERR"]) < 3e-4 and float(kv["ICPCOUNT"]) > 2400 and float(kv["PHOTO"]) < 115, out
    assert float(kv["TDIFF"]) < 0.03 and int(kv["CONSTRAINTS"]) > 10, out
