"""The C++ drop-in classes (host/: feature_matcher, eight_point with the reference's signatures)
built over the C ABI.  CPU part: they compile and link, and without a GPU the driver fails loudly
(there is no CPU fallback).  GPU part: the driver's outputs equal the oracle's."""
import os
import struct
import subprocess

import numpy as np
import pytest

import oracle as O
from erp_match_eightpoint_test_b200 import binding, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "host")
EXE = os.path.join(HOST, "_build", "dropin_main")


def _build():
    from erp_match_eightpoint_test_b200 import build as b

    b.build()
    subprocess.run(["make", "-C", HOST], check=True, capture_output=True)
    assert os.path.exists(EXE)


def _write_input(path, q, t, lxy, rxy, W, H):
    with open(path, "wb") as f:
        f.write(struct.pack("<5i", q.shape[0], t.shape[0], q.shape[1], W, H))
        for a in (q, t, lxy, rxy):
            f.write(np.ascontiguousarray(a, np.float32).tobytes())


def _scene(nq=3000, nt=3200, W=4096, H=2048, seed=21):
    q, t, planted = synth.descriptor_pair(nq, nt, 64, seed=seed)
    qi = np.nonzero(planted >= 0)[0]
    kp = synth.keypoint_pair(len(qi), W, H, noise_px=0.3, outlier_frac=0.0, seed=seed + 1)
    rng = np.random.default_rng(seed)
    lxy = (rng.uniform(0, 1, (nq, 2)) * [W, H - 1]).astype(np.float32)
    rxy = (rng.uniform(0, 1, (nt, 2)) * [W, H - 1]).astype(np.float32)
    lxy[qi] = kp["left_xy"]
    rxy[planted[qi]] = kp["right_xy"]
    return q, t, lxy, rxy, W, H


def test_host_classes_build_and_refuse_to_run_without_a_gpu(tmp_path):
    _build()
    syms = subprocess.run(["nm", "-C", os.path.join(HOST, "_build", "liberp_host.a")], capture_output=True, text=True).stdout
    for name in ["feature_matcher::match_two_image(cv::Mat const&, cv::Mat const&)", "feature_matcher::init()",
                 "feature_matcher::detect_key_point(cv::Mat const&)", "feature_matcher::do_all(",
                 "eight_point::find(int, int, std::vector<cv::KeyPoint", "eight_point::eight_point_estimation(int, int,",
                 "eight_point::initial_guess(int, int,", "random_array::random_array(int)", "erp_rotation::rot2eular(cv::Mat)",
                 "erp_rotation::rotate_image(cv::Mat const&, cv::Mat&)", "erp_rotation::rotate_pixel(",
                 "epipolar_tool::epipolar_tool(std::vector<cv::KeyPoint", "epipolar_tool::draw_epipole(cv::Mat&)",
                 "feature_matcher::set_extended(bool)", "erp_host::write_initial_pose(", "erp_host::read_initial_pose("]:
        assert name in syms, name
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu test")
    q, t, lxy, rxy, W, H = _scene(200, 220)
    inp, out = tmp_path / "in.bin", tmp_path / "out.bin"
    _write_input(inp, q, t, lxy, rxy, W, H)
    r = subprocess.run([EXE, str(inp), str(out)], capture_output=True, text=True)
    assert r.returncode == 1 and "no CPU fallback" in r.stderr and not out.exists()


def test_extrinsic_log_format_and_round_trip(tmp_path):
    """estimated_extrinsic.txt (src/automatic.cpp:135-136): Euler angles in degrees and the unit translation, each as
    "[a, b, c]" with six significant digits; the reader skips the other lines and returns radians."""
    _build()
    exe = os.path.join(HOST, "_build", "log_main")
    r = [0.0872664626, -0.1745329252, 0.2617993878]
    t = [0.3128689, -0.9386067, 0.1042896]
    log = tmp_path / "estimated_extrinsic.txt"
    p = subprocess.run([exe, str(log)] + ["%.10g" % x for x in r + t], capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    lines = open(log).read().splitlines()
    assert lines[0] == "match result"
    assert lines[1] == "initial_R_vector: [%g, %g, %g]" % tuple(180.0 * x / np.pi for x in r)
    assert lines[2] == "initial_T_vector: [%g, %g, %g]" % tuple(t)
    back = [float(x) for x in p.stdout.split()]
    assert np.allclose(back[:3], r, rtol=1e-5) and np.allclose(back[3:], t, rtol=1e-5)      # six significant digits


# The reference's C++ sources are not part of this repository: these tests run when $ERP_REFERENCE_DIR names a checkout
# of Kitsunetic/ERP_match_eightpoint_test.
REFERENCE = os.path.join(os.environ.get("ERP_REFERENCE_DIR", ""), "src")
needs_reference = pytest.mark.skipif(not os.environ.get("ERP_REFERENCE_DIR") or not os.path.isdir(REFERENCE),
                                     reason="set ERP_REFERENCE_DIR to a checkout of the reference project")


@needs_reference
def test_reference_callers_compile_and_link_unchanged(tmp_path):
    """north_star: "automatic.cpp and the test mains link against it unchanged".  The reference's own callers
    (src/automatic.cpp, src/spherical_surf.cpp + .hpp: everything that is NOT replaced) are copied to a scratch
    directory at test time -- next to the reference's headers they would include those instead of the drop-in's -- and
    compiled + linked, unmodified, against host/*.hpp, liberp_host.a and liberp_b200.so (OpenCV: the type shim; the
    only thing this image cannot provide is image codecs, so the binary is linked, not run on images)."""
    _build()
    import shutil
    for f in ("automatic.cpp", "spherical_surf.cpp", "spherical_surf.hpp"):
        shutil.copy(os.path.join(REFERENCE, f), tmp_path / f)
    exe = tmp_path / "automatic.out"
    cmd = ["g++", "-std=c++11", "-O1", "-fopenmp", "-w", f"-I{tmp_path}", f"-I{HOST}", f"-I{HOST}/compat", f"-I{ROOT}/include",
           str(tmp_path / "automatic.cpp"), str(tmp_path / "spherical_surf.cpp"), os.path.join(HOST, "_build", "liberp_host.a"),
           f"-L{ROOT}/erp_match_eightpoint_test_b200/lib", "-lerp_b200", f"-Wl,-rpath,{ROOT}/erp_match_eightpoint_test_b200/lib",
           "-o", str(exe)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    # the classes the callers use resolve to the drop-in's objects
    syms = subprocess.run(["nm", "-C", str(exe)], capture_output=True, text=True).stdout
    for name in ("feature_matcher::match_two_image", "eight_point::find", "erp_rotation::rotate_pixel", "erp_rotation::rotate_image",
                 "spherical_surf::do_all"):
        assert name in syms, name
    usage = subprocess.run([str(exe)], capture_output=True, text=True)
    assert usage.returncode == 0 and "usage:" in usage.stdout
    # manual.cpp and the GUI test mains (one_image_test, image_rotate_test, manual_*_test) need highgui windows,
    # trackbars and mouse callbacks: out of scope; the two-image test mains follow below


@needs_reference
@pytest.mark.parametrize("main_dir", ["two_real_image_test", "two_synthesis_image_test"])
def test_reference_test_mains_compile_and_link_unchanged(tmp_path, main_dir):
    """The reference's own test programs for this path (two_real_image_test/main.cpp: do_all + three find() calls on a real
    pair; two_synthesis_image_test/main.cpp: the same on a rotated copy) compile and link, unmodified, against the drop-in
    classes -- copied to a scratch directory at test time together with the reference files that are NOT replaced."""
    _build()
    import shutil
    ref_root = os.path.dirname(REFERENCE)
    shutil.copy(os.path.join(ref_root, main_dir, "main.cpp"), tmp_path / "main.cpp")
    for f in ("spherical_surf.cpp", "spherical_surf.hpp", "common_header.hpp", "INIReader.h", "pathkit.hpp"):
        if os.path.exists(os.path.join(REFERENCE, f)):
            shutil.copy(os.path.join(REFERENCE, f), tmp_path / f)
    exe = tmp_path / "main.out"
    cmd = ["g++", "-std=c++11", "-O1", "-fopenmp", "-w", f"-I{tmp_path}", f"-I{HOST}", f"-I{HOST}/compat", f"-I{ROOT}/include",
           str(tmp_path / "main.cpp"), str(tmp_path / "spherical_surf.cpp"), os.path.join(HOST, "_build", "liberp_host.a"),
           f"-L{ROOT}/erp_match_eightpoint_test_b200/lib", "-lerp_b200", f"-Wl,-rpath,{ROOT}/erp_match_eightpoint_test_b200/lib",
           "-o", str(exe)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    syms = subprocess.run(["nm", "-C", str(exe)], capture_output=True, text=True).stdout
    for name in ("feature_matcher::match_two_image", "eight_point::find", "spherical_surf::do_all"):
        assert name in syms, name


def test_rotate_pixel_loops_run_on_the_host(tmp_path):
    """erp_rotation::rotate_pixel per pixel from an OpenMP loop (what spherical_surf::crop_rotated_image does,
    src/spherical_surf.cpp:27-45) at the reference's image size: plain host arithmetic, no CUDA context (this test has
    no GPU), same integers as the oracle, and the whole 5376 x 672 strip well under a second per core-second budget."""
    _build()
    exe = os.path.join(HOST, "_build", "strip_main")
    W, H = 5376, 2688
    for pitch in (45.0, -90.0):
        out = tmp_path / "map.bin"
        r = subprocess.run([exe, str(W), str(H), str(pitch), str(out)], capture_output=True, text=True, timeout=120)
        assert r.returncode == 0, r.stderr
        sec = float(r.stdout.split()[0])
        got = np.fromfile(out, np.int32).reshape(-1, 2)
        rows = H // 4
        rc = np.stack(np.meshgrid(np.arange(H * 3 // 8, H * 3 // 8 + rows), np.arange(W), indexing="ij"), -1).reshape(-1, 2).astype(np.int32)
        want = O.rotate_pixels(rc, O.eular2rot([0.0, float(np.float32(np.pi * pitch / 180.0)), 0.0]), W, H)     # Vec3f angle, as the callers pass it
        assert np.array_equal(got, want)
        threads = int(r.stdout.split()[-2])
        assert sec * threads < 8.0, r.stdout          # ~0.1 us of trigonometry per pixel and thread; a device round trip would be ~20 us


@pytest.mark.gpu
def test_reference_strip_loop_equals_the_device_strip(tmp_path):
    """The same host loop fills a strip from a real-sized image; erp_crop_rotated_image (device) picks the same pixels
    up to the documented libm boundary cases (a mapped coordinate within an ulp of an integer: CUDA libm vs glibc; the
    45-degree strips put many pixel centres on such boundaries, tests/test_gpu_image.py uses the same 2 % bar)."""
    _build()
    exe = os.path.join(HOST, "_build", "strip_main")
    W, H = 5376, 2688
    rng = np.random.default_rng(3)
    im = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    img = tmp_path / "im.bin"
    im.tofile(img)
    r = subprocess.run([exe, str(W), str(H), "45", str(tmp_path / "map.bin"), str(img), str(tmp_path / "strip.bin")],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    sec = float(r.stdout.split()[0])
    assert sec < 1.0, r.stdout
    differ = int(r.stdout.splitlines()[-1].split()[4])
    assert differ <= 2e-2 * (H // 4) * W, r.stdout
    strip = np.fromfile(tmp_path / "strip.bin", np.uint8).reshape(H // 4, W, 3)
    assert np.array_equal(strip, O.crop_rotated_image(im, 45.0))


@pytest.mark.gpu
def test_dropin_driver_matches_oracle(tmp_path):
    _build()
    q, t, lxy, rxy, W, H = _scene()
    inp, out, log = tmp_path / "in.bin", tmp_path / "out.bin", tmp_path / "estimated_extrinsic.txt"
    _write_input(inp, q, t, lxy, rxy, W, H)
    r = subprocess.run([EXE, str(inp), str(out), str(log)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    raw = open(out, "rb").read()
    n = struct.unpack_from("<i", raw, 0)[0]
    got = np.frombuffer(raw, binding.DMATCH, n, 4)
    want = O.match(q, t, 0.3, False)
    assert got.tobytes() == want.tobytes()                       # feature_matcher::match_two_image
    off = 4 + 16 * n
    R = np.frombuffer(raw, np.float32, 3, off); T = np.frombuffer(raw, np.float32, 3, off + 12)
    v = np.frombuffer(raw, np.int32, 2, off + 24)
    R1 = np.frombuffer(raw, np.float32, 3, off + 32); R2 = np.frombuffer(raw, np.float32, 3, off + 44)
    Tn = np.frombuffer(raw, np.float32, 3, off + 56)
    l = O.bearings(lxy[want["queryIdx"]], W, H)
    rr = O.bearings(rxy[want["trainIdx"]], W, H)
    ref = O.initial_guess(l, rr, O.ref_sample_table(n))          # eight_point::find
    assert np.abs(R - ref["R"]).max() < 1e-5 and np.abs(T - ref["T"]).max() < 1e-5
    e = O.eight_point(l[:64], rr[:64])                           # eight_point::eight_point_estimation
    a = np.abs(R1 - e["R1"]).max() + np.abs(R2 - e["R2"]).max()
    b = np.abs(R1 - e["R2"]).max() + np.abs(R2 - e["R1"]).max()
    assert min(a, b) < 2e-5 and np.abs(np.abs(Tn) - np.abs(e["T"])).max() < 1e-5
    assert set(v.tolist()) <= {0, 1}
    # estimated_extrinsic.txt: the two lines of src/automatic.cpp:135-136, degrees then unit translation, "%g" numbers
    deg = [180.0 * float(x) / np.pi for x in R]
    want_log = ("initial_R_vector: [%g, %g, %g]\ninitial_T_vector: [%g, %g, %g]\n"
                % (deg[0], deg[1], deg[2], float(T[0]), float(T[1]), float(T[2])))
    assert open(log).read() == want_log
