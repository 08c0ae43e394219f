"""The stream-K planner of the tcgen05 distance kernels (tc_common.cuh: stream_k_plan, SegIter) run on the host, no GPU.

A small program compiled with the library's nvcc flags prints the plan and every CTA's segments for a grid of shapes,
SM counts and segment limits.  The test checks what the kernels rely on: every (query tile, train tile) unit is scanned
exactly once, a segment never leaves its query row, and no two segments of a row share a candidate list slot.  Two
writers of one slot would overwrite a list and its bound, and the certificate would then hold for the wrong list.  It
also checks that tests/test_gpu_pipeline_plans.py's Python copy of the planner agrees with the real one.
"""
import os
import subprocess

import numpy as np
import pytest

from erp_match_eightpoint_test_b200 import build
from test_gpu_pipeline_plans import seg_iter, stream_k_plan

HARNESS = r"""
#include "tc_common.cuh"
#include <cstdio>
#include <vector>
// stdin: lines "n_rows n_ttiles sms max_seg"; stdout per line: "L n_seg grid n_segments" and one "cta row t0 t1 seg"
// line per segment
int main()
{
    int n_rows, n_ttiles, sms, max_seg;
    while (scanf("%d %d %d %d", &n_rows, &n_ttiles, &sms, &max_seg) == 4) {
        const erp::StreamK p = erp::stream_k_plan(n_rows, n_ttiles, sms, max_seg);
        std::vector<int> segs;
        for (int cta = 0; cta < p.grid; cta++) {
            erp::SegIter it(n_rows, n_ttiles, p.units_per_cta, cta);
            int row, t0, t1, seg;
            while (it.next(row, t0, t1, seg)) segs.insert(segs.end(), {cta, row, t0, t1, seg});
        }
        printf("%d %d %d %zu\n", p.units_per_cta, p.n_seg, p.grid, segs.size() / 5);
        for (size_t i = 0; i < segs.size(); i += 5) printf("%d %d %d %d %d\n", segs[i], segs[i + 1], segs[i + 2], segs[i + 3], segs[i + 4]);
    }
    return 0;
}
"""

# 1..800 query rows (units) and train tiles: every small value, the values around the segment limits and the SM
# counts, and large ones
SIZES = sorted(set(range(1, 18)) | {29, 31, 32, 33, 63, 64, 100, 127, 131, 132, 133, 147, 148, 149, 255, 257, 296, 500, 799, 800})
SMS = (1, 7, 132, 148)
MAX_SEGS = (8, 16)               # distance kernels of float rows (F_MAX_SEG, MAX_SEG) and of binary rows (B_MAX_SEG)
TOPK = 8                         # the widest float candidate list (knn_tc1.cu F_TOPK), two column groups per segment


@pytest.fixture(scope="module")
def dump(tmp_path_factory):
    if not os.path.exists(build.NVCC):
        pytest.skip("nvcc not found")
    d = tmp_path_factory.mktemp("plan")
    src, exe = d / "plan_dump.cu", d / "plan_dump"
    src.write_text(HARNESS)
    r = subprocess.run([build.NVCC] + build.FLAGS + [str(src), "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    shapes = [(nr, nt, sms, ms) for sms in SMS for ms in MAX_SEGS for nr in SIZES for nt in SIZES]
    r = subprocess.run([str(exe)], input="".join("%d %d %d %d\n" % s for s in shapes), capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    vals = np.fromstring(r.stdout, np.int64, sep=" ")
    out, k = [], 0
    for s in shapes:
        L, n_seg, grid, n = vals[k: k + 4]
        out.append((s, (int(L), int(n_seg), int(grid)), vals[k + 4: k + 4 + 5 * n].reshape(n, 5)))
        k += 4 + 5 * n
    assert k == len(vals)
    return out


def test_plan_covers_every_unit_once_and_never_shares_a_list_slot(dump):
    for (n_rows, n_ttiles, sms, max_seg), (L, n_seg, grid), segs in dump:
        ctx = (n_rows, n_ttiles, sms, max_seg, L, n_seg, grid)
        total = n_rows * n_ttiles
        cta, row, t0, t1, seg = segs.T
        assert (grid - 1) * L < total <= grid * L, ctx
        assert 2 <= n_seg <= max_seg - 1, ctx
        if max_seg == 8:
            assert n_seg * 2 * TOPK <= 128, ctx               # refine_launch holds 128 candidate slots per query
        # a segment is a non-empty run of train tiles inside one query row
        assert ((0 <= row) & (row < n_rows) & (0 <= t0) & (t0 < t1) & (t1 <= n_ttiles)).all(), ctx
        # in CTA order the segments tile the unit range [0, total) without gap or overlap, each inside its CTA's range
        u0, u1 = row * n_ttiles + t0, row * n_ttiles + t1
        assert u0[0] == 0 and u1[-1] == total and (u0[1:] == u1[:-1]).all(), ctx
        assert ((cta * L <= u0) & (u1 <= cta * L + L)).all() and (np.diff(cta) >= 0).all(), ctx
        # the list slot: inside [0, n_seg), and one writer per (row, slot)
        assert ((0 <= seg) & (seg < n_seg)).all(), ctx
        assert len(np.unique(row * max_seg + seg)) == len(seg), ctx


def test_python_mirror_equals_the_planner(dump):
    for (n_rows, n_ttiles, sms, max_seg), plan, segs in dump:
        L, n_seg, grid = stream_k_plan(n_rows, n_ttiles, sms, max_seg)
        assert (L, n_seg, grid) == plan, (n_rows, n_ttiles, sms, max_seg)
        mirror = [(c,) + s for c in range(grid) for s in seg_iter(n_rows, n_ttiles, L, c)]
        assert np.array_equal(np.array(mirror, np.int64).reshape(-1, 5), segs), (n_rows, n_ttiles, sms, max_seg)
