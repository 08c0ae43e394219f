"""CPU reference of Hamming 2-NN matching (cv::BFMatcher(NORM_HAMMING) semantics), brute force with numpy popcounts.

knn2: the two nearest train rows of every query in (distance, trainIdx) order; match: ratio test in fp32
(d0 < ratio * d1, ratio < 0 disables it), cross-check (mutual nearest, reverse ties to the lowest queryIdx), records in
ascending queryIdx, the layout of erp_dmatch.
"""
from __future__ import annotations

import numpy as np

DMATCH = np.dtype([("queryIdx", "<i4"), ("trainIdx", "<i4"), ("imgIdx", "<i4"), ("distance", "<f4")])


def _words(a: np.ndarray) -> np.ndarray:
    a = np.ascontiguousarray(a, np.uint8)
    pad = (-a.shape[1]) % 8
    if pad:
        a = np.concatenate([a, np.zeros((a.shape[0], pad), np.uint8)], axis=1)
    return a.view(np.uint64)


def distances(q: np.ndarray, t: np.ndarray) -> np.ndarray:
    """Full nq x nt Hamming distance matrix (int32)."""
    qw, tw = _words(q), _words(t)
    return np.bitwise_count(qw[:, None, :] ^ tw[None, :, :]).sum(axis=2, dtype=np.int32)


def knn2(q: np.ndarray, t: np.ndarray, chunk: int = 256):
    """(idx (nq, 2) int32, dist (nq, 2) float32); a missing second neighbour is -1 / inf."""
    nq, nt = q.shape[0], t.shape[0]
    idx = np.full((nq, 2), -1, np.int32)
    dist = np.full((nq, 2), np.inf, np.float32)
    tw = _words(t)
    qw_all = _words(q)
    rows = np.arange(chunk)
    for s in range(0, nq, chunk):
        qw = qw_all[s:s + chunk]
        d = np.bitwise_count(qw[:, None, :] ^ tw[None, :, :]).sum(axis=2, dtype=np.int32)
        r = rows[: d.shape[0]]
        i0 = np.argmin(d, axis=1)            # first occurrence: the lowest index among equal distances
        idx[s:s + len(r), 0] = i0
        dist[s:s + len(r), 0] = d[r, i0]
        if nt >= 2:
            d[r, i0] = np.iinfo(np.int32).max
            i1 = np.argmin(d, axis=1)
            idx[s:s + len(r), 1] = i1
            dist[s:s + len(r), 1] = d[r, i1]
    return idx, dist


def match(q: np.ndarray, t: np.ndarray, ratio: float = 0.8, cross_check: bool = False, knn=None) -> np.ndarray:
    idx, dist = knn2(q, t) if knn is None else knn
    keep = idx[:, 0] >= 0
    if ratio >= 0:
        keep &= dist[:, 0] < np.float32(ratio) * dist[:, 1]
    if cross_check:
        rev = knn2(t, q)[0][:, 0]
        keep &= rev[np.maximum(idx[:, 0], 0)] == np.arange(len(q))
    qi = np.nonzero(keep)[0]
    out = np.zeros(len(qi), DMATCH)
    out["queryIdx"] = qi
    out["trainIdx"] = idx[qi, 0]
    out["distance"] = dist[qi, 0]
    return out


# A caller of the drop-in feature_matcher with norm_type = cv::NORM_HAMMING: reads nq, nt, nbytes, the two uint8 row
# blocks and (ratio, cross_check), writes n and the DMatch records.  The default norm_type must refuse CV_8U rows.
HAMMING_MAIN = r"""
#include <cstdio>
#include <vector>
#include "feature_matcher.hpp"
int main(int argc, char** argv)
{
    if (argc != 3) return 2;
    FILE* f = fopen(argv[1], "rb");
    int h[3]; float ratio; int cc;
    if (fread(h, 4, 3, f) != 3) return 2;
    std::vector<unsigned char> q((size_t)h[0] * h[2]), t((size_t)h[1] * h[2]);
    if (fread(q.data(), 1, q.size(), f) != q.size() || fread(t.data(), 1, t.size(), f) != t.size()) return 2;
    if (fread(&ratio, 4, 1, f) != 1 || fread(&cc, 4, 1, f) != 1) return 2;
    fclose(f);
    cv::Mat dq(h[0], h[2], CV_8UC1, q.data()), dt(h[1], h[2], CV_8UC1, t.data());
    feature_matcher fm;
    if (fm.norm_type != cv::NORM_L2) return 3;
    try { fm.match_two_image(dq, dt); return 4; } catch (const cv::Exception&) {}
    fm.norm_type = cv::NORM_HAMMING;
    fm.ratio_thresh = ratio;
    fm.cross_check = cc != 0;
    std::vector<cv::DMatch> m;
    try { m = fm.match_two_image(dq, dt); }
    catch (const std::exception& e) { fprintf(stderr, "%s\n", e.what()); return 1; }
    FILE* o = fopen(argv[2], "wb");
    int n = (int)m.size();
    fwrite(&n, 4, 1, o);
    fwrite(m.data(), sizeof(cv::DMatch), m.size(), o);
    fclose(o);
    return 0;
}
"""


def build_hamming_main(tmp_path):
    """Builds the library, the host classes and HAMMING_MAIN; returns the executable's path."""
    import os
    import subprocess

    from erp_match_eightpoint_test_b200 import build as b

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    host = os.path.join(root, "host")
    b.build()
    subprocess.run(["make", "-C", host], check=True, capture_output=True)
    src, exe = tmp_path / "hamming_main.cpp", tmp_path / "hamming_main"
    src.write_text(HAMMING_MAIN)
    cmd = ["g++", "-std=c++17", "-O1", f"-I{host}", f"-I{host}/compat", f"-I{root}/include", str(src),
           os.path.join(host, "_build", "liberp_host.a"), f"-L{root}/erp_match_eightpoint_test_b200/lib", "-lerp_b200",
           f"-Wl,-rpath,{root}/erp_match_eightpoint_test_b200/lib", "-o", str(exe)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return exe


def write_hamming_input(path, q, t, ratio, cross_check):
    with open(path, "wb") as f:
        f.write(np.array([q.shape[0], t.shape[0], q.shape[1]], np.int32).tobytes())
        f.write(np.ascontiguousarray(q, np.uint8).tobytes())
        f.write(np.ascontiguousarray(t, np.uint8).tobytes())
        f.write(np.array([ratio], np.float32).tobytes() + np.array([int(cross_check)], np.int32).tobytes())


def read_hamming_output(path):
    raw = open(path, "rb").read()
    n = int(np.frombuffer(raw[:4], np.int32)[0])
    return np.frombuffer(raw[4:4 + 16 * n], DMATCH)
