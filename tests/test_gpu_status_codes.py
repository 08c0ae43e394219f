"""Status codes of the match and pair entry points for every bad input their checks reject: float and binary rows, host and
device forms, and the multi-GPU forms on a context without a clique (which answer like the one-GPU calls, apart from
erp_knn2_match_dist_dev, which checks on its own).  The order of the checks is pinned too: an input that breaks two rules
gets the status of the rule checked first."""
import ctypes as C

import numpy as np
import pytest

import erp_match_eightpoint_test_b200 as erp
from erp_match_eightpoint_test_b200 import binding as B

pytestmark = pytest.mark.gpu

NQ, NT, DIM, NBYTES = 64, 64, 64, 32
FW, BW = 256, 64                     # host row pitch of the float (in floats) and binary (in bytes) descriptors
IMG_W, IMG_H = 1024, 512
NULL = object()                      # an override that passes a null pointer

# entry -> (row kind, form, arguments in the order of the C ABI); a name stands for the value of that key
ENTRIES = {
    "erp_knn2_dev": ("f32", "dev", "ctx q nq t nt dim idx dist d2"),
    "erp_knn2_bin_dev": ("bin", "dev", "ctx q nq t nt dim idx dist d2"),
    "erp_nn1_reverse_dev": ("f32", "dev", "ctx q nq t nt dim zero rev d2"),
    "erp_knn2_match_dev": ("f32", "dev", "ctx q nq t nt dim ratio cross out n"),
    "erp_knn2_match_bin_dev": ("bin", "dev", "ctx q nq t nt dim ratio cross out n"),
    "erp_knn2_match_dist_dev": ("f32", "dev", "ctx q nq t nt dim ratio cross out n"),
    "erp_knn2_match": ("f32", "host", "ctx q nq qs t nt ts dim ratio cross out n"),
    "erp_knn2_match_bin": ("bin", "host", "ctx q nq qs t nt ts dim ratio cross out n"),
    "erp_knn2_match_dist": ("f32", "host", "ctx q nq qs t nt ts dim ratio cross out n"),
    "erp_knn2_raw": ("f32", "host", "ctx q nq qs t nt ts dim idx dist"),
    "erp_knn2_raw_bin": ("bin", "host", "ctx q nq qs t nt ts dim idx dist"),
    "erp_knn2_near_ties": ("f32", "host", "ctx q nq qs t nt ts dim tol flags n"),
    "erp_pair_pose_dev": ("f32", "dev", "ctx q nq t nt dim ratio cross l r kps w h seed H S metric tau out n mask res"),
    "erp_pair_pose_bin_dev": ("bin", "dev", "ctx q nq t nt dim ratio cross l r kps w h seed H S metric tau out n mask res"),
    "erp_pair_pose_dist_dev": ("f32", "dev", "ctx q nq t nt dim ratio cross l r kps w h seed H S metric tau out n mask res"),
    "erp_pair_pose": ("f32", "host", "ctx q nq qs t nt ts dim ratio cross l r kps w h seed H S metric tau out n res mask"),
    "erp_pair_pose_bin": ("bin", "host", "ctx q nq qs t nt ts dim ratio cross l r kps w h seed H S metric tau out n res mask"),
    "erp_pair_pose_dist": ("f32", "host", "ctx q nq qs t nt ts dim ratio cross l r kps w h seed H S metric tau out n res mask"),
}
PAIR = {e for e in ENTRIES if "pair_pose" in e}
MATCH = set(ENTRIES) - PAIR - {"erp_nn1_reverse_dev"}

# the size and dimension rules every match and pair entry shares
KNN_CASES = [
    ("null context", dict(ctx=NULL), B.E_ARG),
    ("nq < 0", dict(nq=-1), B.E_ARG),
    ("nt < 0", dict(nt=-1), B.E_ARG),
    ("dim 0", dict(dim=0), B.E_DIM),
    ("nt 1", dict(nt=1), B.E_TOO_FEW_TRAIN),
    ("nt 1 and dim 0", dict(nt=1, dim=0), B.E_DIM),
    ("nq < 0 and dim 0", dict(nq=-1, dim=0), B.E_ARG),
]
F32_DIM_CASES = [("dim 6", dict(dim=6), B.E_DIM), ("dim 516", dict(dim=516), B.E_DIM)]
BIN_DIM_CASES = [("nbytes 65", dict(dim=65), B.E_DIM)]
# a tensor engine forced on a shape it cannot serve (float rows of more than 128 values)
FORCED = ("forced tcgen05 at dim 256", dict(engine=B.ENGINE_TCGEN05, dim=256), B.E_DIM)
PAIR_CASES = [
    ("H 0", dict(H=0), B.E_ARG),
    ("S 7", dict(S=7), B.E_ARG),
    ("S 33", dict(S=33), B.E_ARG),
    ("metric 3", dict(metric=3), B.E_ARG),
    ("width 0", dict(w=0), B.E_ARG),
    ("null matches", dict(out=NULL), B.E_ARG),
    ("null match count", dict(n=NULL), B.E_ARG),
    ("null result", dict(res=NULL), B.E_ARG),
    ("null left keypoints", dict(l=NULL), B.E_ARG),
    ("keypoint stride 4", dict(kps=4), B.E_ARG),
    ("keypoint stride 10", dict(kps=10), B.E_ARG),
    ("nq 0", dict(nq=0), B.E_TOO_FEW_POINTS),
    ("nq 0 and H 0", dict(nq=0, H=0), B.E_ARG),
    ("nt 1 and S 7", dict(nt=1, S=7), B.E_TOO_FEW_TRAIN),
    ("dim 0 and H 0", dict(dim=0, H=0), B.E_DIM),
    ("null query rows", dict(q=NULL), B.E_ARG),
    FORCED,
]


def _cases():
    out = []
    for entry, (kind, form, _) in ENTRIES.items():
        if entry == "erp_nn1_reverse_dev":
            cases = [("null context", dict(ctx=NULL), B.E_ARG), ("nq 0", dict(nq=0), B.E_ARG), ("nt < 0", dict(nt=-1), B.E_ARG),
                     ("null best_q", dict(rev=NULL), B.E_ARG), ("dim 6", dict(dim=6), B.E_DIM), ("nq 0 and dim 6", dict(nq=0, dim=6), B.E_ARG)]
        else:
            cases = KNN_CASES + (F32_DIM_CASES if kind == "f32" else BIN_DIM_CASES)
        if entry in MATCH:
            cases = cases + [("null query rows", dict(q=NULL), B.E_ARG)]
            if "n" in ENTRIES[entry][2].split():
                # erp_knn2_match_dist_dev checks its count pointer before the sizes, the others after them
                cases = cases + [("null count", dict(n=NULL), B.E_ARG),
                                 ("null count and nt 1", dict(n=NULL, nt=1),
                                  B.E_ARG if entry == "erp_knn2_match_dist_dev" else B.E_TOO_FEW_TRAIN)]
            if form == "host":
                cases = cases + [("query stride below a row", dict(qs="short"), B.E_ARG)]
            if kind == "f32":
                cases = cases + [FORCED]
        if entry in PAIR:
            cases = cases + PAIR_CASES[:-1] + ([FORCED] if kind == "f32" else [])
            if form == "host":
                cases = cases + [("query stride below a row", dict(qs="short"), B.E_ARG),
                                 ("fewer matches than S", dict(ratio=1e-9), B.E_TOO_FEW_POINTS)]
        if entry in ("erp_knn2_match", "erp_knn2_match_bin", "erp_knn2_match_dist"):
            cases = cases + [("null records", dict(out=NULL), B.E_ARG)]
        if entry == "erp_knn2_near_ties":
            cases = cases + [("negative tolerance", dict(tol=-1.0), B.E_ARG), ("null flags", dict(flags=NULL), B.E_ARG)]
        out += [pytest.param(entry, o, want, id=f"{entry}-{name}") for name, o, want in cases]
    return out


@pytest.fixture(scope="module")
def bufs():
    import torch

    ctx = erp.Context(0)
    rng = np.random.default_rng(5)
    dev = lambda n, dt: torch.zeros(n, dtype=dt, device="cuda")
    b = dict(ctx=ctx)
    b["f32", "host"] = (rng.standard_normal((NQ, FW)).astype(np.float32), rng.standard_normal((NT, FW)).astype(np.float32))
    b["bin", "host"] = (rng.integers(0, 256, (NQ, BW), dtype=np.uint8), rng.integers(0, 256, (NT, BW), dtype=np.uint8))
    b["f32", "dev"] = tuple(torch.from_numpy(a).cuda() for a in b["f32", "host"])
    b["bin", "dev"] = tuple(torch.from_numpy(a).cuda() for a in b["bin", "host"])
    xy = lambda n: (rng.uniform(0, 1, (n, 4)) * [IMG_W, IMG_H - 1, IMG_W, IMG_H - 1]).astype(np.float32)
    b["host_out"] = dict(l=xy(NQ), r=xy(NT), out=np.zeros(NQ, B.DMATCH), idx=np.zeros((NQ, 2), np.int32),
                         dist=np.zeros((NQ, 2), np.float32), flags=np.zeros(NQ, np.uint8), mask=np.zeros(NQ, np.uint8))
    b["dev_out"] = dict(l=torch.from_numpy(b["host_out"]["l"]).cuda(), r=torch.from_numpy(b["host_out"]["r"]).cuda(),
                        out=dev(NQ * 16, torch.uint8), n=dev(4, torch.int32), idx=dev(NQ * 2, torch.int32), dist=dev(NQ * 2, torch.float32),
                        d2=dev(NQ * 2, torch.float64), rev=dev(NT, torch.int32), mask=dev(NQ, torch.uint8), res=dev(512, torch.uint8))
    yield b
    ctx.close()


def _args(b, entry, over):
    kind, form, names = ENTRIES[entry]
    q, t = b[kind, form]
    pitch = q.shape[1] * (4 if kind == "f32" else 1)
    v = dict(ctx=b["ctx"]._h, q=q, t=t, nq=NQ, nt=NT, dim=DIM if kind == "f32" else NBYTES, qs=pitch, ts=pitch, ratio=0.8, cross=1,
             kps=16, w=IMG_W, h=IMG_H, seed=1, H=64, S=8, metric=0, tau=0.002, tol=1e-6, zero=0)
    v.update(b["host_out" if form == "host" else "dev_out"])
    if form == "host":
        v["n"] = C.byref(C.c_int(0))
        v["res"] = C.byref(B.RansacResult())
    v.update(over)
    if v["qs"] == "short":                        # one byte short of a row
        v["qs"] = pitch // q.shape[1] * v["dim"] - 1
    out = []
    for name in names.split():
        x = v[name]
        out.append(None if x is NULL else B._ptr(x) if isinstance(x, np.ndarray) or hasattr(x, "data_ptr") else x)
    return out


@pytest.mark.parametrize("entry,over,want", _cases())
def test_status_code(bufs, entry, over, want):
    over = dict(over)
    engine = over.pop("engine", B.ENGINE_AUTO)
    bufs["ctx"].set_engine(engine)
    try:
        got = getattr(B.lib(), entry)(*_args(bufs, entry, over))
    finally:
        bufs["ctx"].set_engine(B.ENGINE_AUTO)
    assert got == want, B.lib().erp_last_error().decode()
