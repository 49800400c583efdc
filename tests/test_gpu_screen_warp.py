"""The two shapes of the mma.sync screening pass (csrc/dune_screen_mma_kernel.cuh) -- one warp per (environment, step) item
(dune_screen_warp_kernel, the default) and one CTA of four warps per item (dune_screen_mma_kernel, NB_SCREEN_MMA=2) -- compared item by
item on the same inputs: the same candidate SET with the same screened distances, the same counts, the same items flagged for the
exact kernel and the same refine lists.  Only the order inside a candidate list may differ (the refine kernel ranks by distance and
index).  tests/screen_shapes_harness.cu runs one kernel on host arrays; it is compiled here against the built library."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from helpers import CONFIGS, weights_path
from neupan_b200 import _lib
from neupan_b200 import build as nb_build

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
KCAND = 32


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    lib_path = nb_build.build()
    out = str(tmp_path_factory.mktemp("screen_harness") / "screen_shapes_harness.so")
    libdir = os.path.dirname(lib_path)
    cmd = [nb_build._nvcc(), *nb_build.ARCH, "-O3", "-std=c++17", "-shared", "-Xcompiler", "-fPIC", "-I", nb_build.CSRC,
           os.path.join(HERE, "screen_shapes_harness.cu"), "-o", out, "-L", libdir, "-lneupan_b200", f"-Xlinker=-rpath={libdir}"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    _lib.load()  # the library the harness links against, already loaded with its dependencies
    h = C.CDLL(out)
    h.nb_test_screen.restype = C.c_int
    return h


def _weights(model):
    z = np.load(weights_path(model))
    return np.concatenate([np.ascontiguousarray(z[f"MLP.{i}.{k}"], np.float32).reshape(-1)
                           for i in (0, 1, 3, 5, 6, 8, 10, 11, 13) for k in ("weight", "bias")])


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _screen(h, shape, cfg, inp, N, c_mu, skip_t0=0, calibrate=0, num_points=None, active=None):
    rb = cfg.make_robot()
    G = np.ascontiguousarray(np.asarray(rb.G), np.float32)
    hv = np.ascontiguousarray(np.asarray(rb.h), np.float32).reshape(-1)
    B, T, M, E = inp["points"].shape[0], cfg.T, cfg.M, G.shape[0]
    items = B * (T + 1)
    out = dict(cand_idx=np.empty((items, KCAND), np.int32), cand_dt=np.empty((items, KCAND), np.float32), cand_cnt=np.empty(items, np.int32),
               flag_list=np.empty(items, np.int32), refine_list=np.empty(2 * items, np.int32), flag_count=np.empty(4, np.int32),
               stats=np.empty(4, np.uint32), sel_count=np.empty(B, np.int32), min_dist=np.empty(B, np.float32))
    f32 = lambda k: None if inp.get(k) is None else np.ascontiguousarray(inp[k], np.float32)
    w = _weights(cfg.model)
    rc = h.nb_test_screen(shape, B, N, T, M, E, _ptr(G), _ptr(hv), C.c_float(c_mu), C.c_float(cfg.dt), skip_t0, calibrate,
                          _ptr(f32("nom_s")), _ptr(f32("points")), _ptr(f32("velocities")), _ptr(num_points), _ptr(active), _ptr(w),
                          *[_ptr(out[k]) for k in ("cand_idx", "cand_dt", "cand_cnt", "flag_list", "refine_list", "flag_count", "stats",
                                                   "sel_count", "min_dist")])
    assert rc == 0, rc
    return out


def _assert_same_screen(a, b):
    items = a["cand_cnt"].size
    assert np.array_equal(a["cand_cnt"], b["cand_cnt"])
    for it in np.nonzero(a["cand_cnt"] > 0)[0]:
        c = a["cand_cnt"][it]
        oa, ob = np.argsort(a["cand_idx"][it, :c], kind="stable"), np.argsort(b["cand_idx"][it, :c], kind="stable")
        assert np.array_equal(a["cand_idx"][it, :c][oa], b["cand_idx"][it, :c][ob]), it
        assert np.array_equal(a["cand_dt"][it, :c][oa].view(np.int32), b["cand_dt"][it, :c][ob].view(np.int32)), it
    assert np.array_equal(a["flag_count"][:3], b["flag_count"][:3])
    nf = a["flag_count"][0]
    assert np.array_equal(np.sort(a["flag_list"][:nf]), np.sort(b["flag_list"][:nf]))
    assert np.array_equal(np.nonzero(a["cand_cnt"] == -1)[0], np.sort(a["flag_list"][:nf]))
    for cls, n in ((0, a["flag_count"][1]), (1, a["flag_count"][2])):
        ra, rb = a["refine_list"][cls * items:cls * items + n], b["refine_list"][cls * items:cls * items + n]
        assert np.array_equal(np.sort(ra), np.sort(rb))
    assert np.array_equal(a["stats"][1:], b["stats"][1:])
    assert np.array_equal(a["sel_count"], b["sel_count"])
    assert np.array_equal(a["min_dist"].view(np.int32), b["min_dist"].view(np.int32))


@pytest.mark.parametrize("c_mu", [0.01, 0.06])
@pytest.mark.parametrize("scene", ["annulus", "obstacles"])
@pytest.mark.parametrize("cname", ["C2", "C4", "C5"])
def test_warp_and_cta_shapes_give_the_same_candidates(harness, cname, scene, c_mu):
    from neupan_b200.synth import make_inputs

    cfg = CONFIGS[cname]
    inp = make_inputs(cfg, B=64, scene=scene)
    warp, cta = (_screen(harness, s, cfg, inp, cfg.N, c_mu) for s in (1, 2))
    _assert_same_screen(warp, cta)
    screened, flagged = warp["stats"][3], warp["stats"][1]
    if c_mu < 0.05:
        assert screened > 0
    else:
        assert flagged > 0  # a wide bound overflows candidate lists (in some scenes all of them): that path is compared too


@pytest.mark.parametrize("cname", ["C2", "C4", "C5"])
def test_shapes_agree_on_ragged_stopped_skipped_and_calibration_items(harness, cname):
    from neupan_b200.synth import make_inputs

    cfg = CONFIGS[cname]
    B = 12
    inp = make_inputs(cfg, B=B, scene="obstacles")
    N = cfg.N
    counts = np.array([N, 0, 5, 33, N // 2, 32, 31, 1, 64, 65, N - 1, 10][:B], np.int32)
    active = np.array([1, 1, 1, 1, 0, 1, 1, 1, 1, 0, 1, 1][:B], np.int32)
    for kw in (dict(num_points=counts, active=active), dict(num_points=counts, skip_t0=1), dict(skip_t0=1, active=active)):
        warp, cta = (_screen(harness, s, cfg, inp, N, 0.02, **kw) for s in (1, 2))
        _assert_same_screen(warp, cta)
    # calibration mode: clouds of <= 32 points are screened too, every point becomes a candidate with its screened distance
    small = make_inputs(cfg, B=B, N=32, scene="obstacles")
    warp, cta = (_screen(harness, s, cfg, small, 32, 0.02, calibrate=1, num_points=np.minimum(counts, 32)) for s in (1, 2))
    _assert_same_screen(warp, cta)
    assert np.isfinite(warp["cand_dt"][warp["cand_cnt"] > 0, 0]).all()
