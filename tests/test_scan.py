"""Lidar scan -> points (SURVEY 8f "next" row 2): oracle vs the reference's golden vectors (CPU), CUDA kernel vs both (GPU)."""
import importlib.util
import os

import numpy as np
import pytest

from oracle import scan as oscan

HERE = os.path.dirname(os.path.abspath(__file__))
_spec = importlib.util.spec_from_file_location("make_golden_scan", os.path.join(HERE, "golden", "make_golden_scan.py"))
mgs = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(mgs)
GOLD = np.load(os.path.join(HERE, "golden", "ref_scan.npz"))
CASES = mgs.CASES


def _case(name):
    B, R, scan, off, ar, ds, mp, vm = CASES[name]
    g = {k.split(".", 1)[1]: GOLD[k] for k in GOLD.files if k.startswith(name + ".")}
    return (B, R, scan, off, ar, ds, mp, vm), g


@pytest.mark.parametrize("name", list(CASES))
def test_oracle_reproduces_reference_golden_vectors(name):
    """oracle/scan.py (per-beam restatement) == outputs of the reference's own functions, bit for bit."""
    (B, R, scan, off, ar, ds, mp, vm), g = _case(name)
    pts, vel, cnt = oscan.scan_batch(g["states"], g["ranges"], scan, off, ar, ds, mp, g["velocity"] if vm else None, vm)
    assert np.array_equal(cnt, g["counts"])
    assert np.array_equal(pts, g["points"])
    if vm:
        assert np.array_equal(vel, g["vel_out"])


def test_golden_vectors_are_current():
    """The reference's scan_to_point_velocity, replayed from its recorded calls (ref_calls.npz) on the fixture's inputs, packed
    by oracle.scan.scan_batch, gives the committed fixture."""
    calls = np.load(os.path.join(HERE, "golden", "ref_calls.npz"))
    (B, R, scan, off, ar, ds, mp, vm), g = _case("velocity_stride")
    seen = []

    def fn_v(st, sc, o, a, d):
        i = len(seen)
        seen.append(i)
        assert np.array_equal(st, calls[f"scan.{i}.state"]) and np.array_equal(sc["ranges"], calls[f"scan.{i}.ranges"])
        assert np.array_equal(sc["velocity"], calls[f"scan.{i}.velocity"])
        return calls[f"scan.{i}.points"], calls[f"scan.{i}.vel"]

    pts, vel, cnt = oscan.scan_batch(g["states"], g["ranges"], scan, off, ar, ds, mp, g["velocity"], True, fn_velocity=fn_v)
    assert len(seen) == int(calls["scan.calls"])
    assert np.array_equal(pts, g["points"]) and np.array_equal(vel, g["vel_out"]) and np.array_equal(cnt, g["counts"])


def test_facade_host_methods_match_oracle():
    """The single-env numpy methods of the planner facade (reference API) agree with the per-beam restatement."""
    from neupan_b200.neupan import neupan as Planner

    (B, R, scan, off, ar, ds, mp, vm), g = _case("velocity_stride")
    fake = Planner.__new__(Planner)
    for b in range(B):
        sc = dict(scan, ranges=g["ranges"][b].astype(float), velocity=g["velocity"][b].astype(float))
        st = g["states"][b].reshape(3, 1)
        p0 = oscan.scan_to_point(st, sc, off, ar, ds)
        p1, v1 = oscan.scan_to_point_velocity(st, sc, off, ar, ds)
        q0 = Planner.scan_to_point(fake, st, sc, list(off), list(ar), ds)
        q1, w1 = Planner.scan_to_point_velocity(fake, st, sc, list(off), list(ar), ds)
        assert np.allclose(p0, q0, rtol=0, atol=1e-12) and np.allclose(p1, q1, rtol=0, atol=1e-12) and np.array_equal(v1, w1)
        assert p0.shape[1] < p1.shape[1]  # the beams exactly at range_min separate the two functions


def test_decimation_map_is_numpy_linspace():
    for n, m in ((307, 100), (720, 100), (334, 64), (101, 100), (5, 1)):
        idx = np.linspace(0, n - 1, m).astype(int)
        step = (n - 1) / (m - 1) if m > 1 else 0.0
        mine = [n - 1 if (j == m - 1 and m > 1) else int(j * step + 0.0) for j in range(m)]
        assert list(idx) == mine  # the formula the kernel evaluates in FP64 (scan_kernel.cuh: linspace_at)


# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_kernel_matches_reference_golden_vectors(name):
    """nb_scan_to_points through the C ABI vs the reference's outputs.  Counts and the beam selection are exact; the
    coordinates go through cos/sin in FP64 on both sides and a float32 cast: tolerance 1 float32 ulp of the value
    (CUDA's FP64 cos/sin are within 2 ulp of libm's, which can flip the last float32 bit)."""
    import torch

    from neupan_b200 import scan_to_points

    (B, R, scan, off, ar, ds, mp, vm), g = _case(name)
    pts, vel, cnt = scan_to_points(torch.from_numpy(g["states"]), torch.from_numpy(g["ranges"]), scan, off, ar, ds, mp,
                                   torch.from_numpy(g["velocity"]) if vm else None, vm)
    cnt = cnt.cpu().numpy()
    assert np.array_equal(cnt, g["counts"])
    got, want = pts.cpu().numpy(), g["points"]
    for b in range(B):
        a, w = got[b, :, :cnt[b]], want[b, :, :cnt[b]]
        assert np.all(np.abs(a - w) <= np.spacing(np.abs(w).astype(np.float32))), (name, b, np.abs(a - w).max())
        if vm:
            assert np.array_equal(vel.cpu().numpy()[b, :, :cnt[b]], g["vel_out"][b, :, :cnt[b]])  # pure gather: exact


@pytest.mark.gpu
@pytest.mark.parametrize("R,mp,ds,vm", [(9000, 300, 1, True), (8192, 8192, 2, False), (40, 40, 1, True), (33, 7, 1, False), (2049, 500, 3, True)])
def test_kernel_matches_oracle_at_other_beam_counts(R, mp, ds, vm):
    """R = 9000 runs the chunked (generic) kernel, the others the register-resident one at 128 ... 1024 threads."""
    import torch

    from neupan_b200 import scan_to_points

    B = 2
    rng = np.random.default_rng(R)
    scan = dict(angle_min=-3.0, angle_max=3.1, range_min=0.3, range_max=9.0)
    ranges = rng.uniform(0.0, 10.0, size=(B, R)).astype(np.float32)
    velocity = rng.normal(size=(B, 2, R)).astype(np.float32)
    states = np.stack([rng.uniform(-5, 5, B), rng.uniform(-5, 5, B), rng.uniform(-np.pi, np.pi, B)], 1)
    off, ar = (0.2, -0.3, 0.5), (-2.9, 3.0)
    want_p, want_v, want_c = oscan.scan_batch(states, ranges, scan, off, ar, ds, mp, velocity if vm else None, vm)
    pts, vel, cnt = scan_to_points(torch.from_numpy(states), torch.from_numpy(ranges), scan, off, ar, ds, mp, torch.from_numpy(velocity) if vm else None, vm)
    cnt = cnt.cpu().numpy()
    assert np.array_equal(cnt, want_c)
    for b in range(B):
        a, w = pts.cpu().numpy()[b, :, :cnt[b]], want_p[b, :, :cnt[b]]
        assert np.all(np.abs(a - w) <= np.spacing(np.abs(w).astype(np.float32)))
        if vm:
            assert np.array_equal(vel.cpu().numpy()[b, :, :cnt[b]], want_v[b, :, :cnt[b]])


@pytest.mark.gpu
def test_kernel_output_feeds_pan_forward_like_the_host_path():
    """scan -> points on the GPU -> PAN.forward(num_points=counts) == host scan_to_point_velocity -> PAN.forward per env."""
    import dataclasses

    import torch

    from gpu_helpers import make_pan
    from helpers import CONFIGS, make_inputs
    from neupan_b200 import scan_to_points

    cfg = dataclasses.replace(CONFIGS["C4"], K=1)
    B, R, mp = 5, 400, 128
    inp = make_inputs(cfg, B=B, N=mp)
    rng = np.random.default_rng(7)
    scan = dict(angle_min=-np.pi, angle_max=np.pi, range_min=0.1, range_max=10.0)
    ranges = rng.uniform(1.5, 11.0, size=(B, R)).astype(np.float32)
    velocity = rng.uniform(-1, 1, size=(B, 2, R)).astype(np.float32)
    states = inp["nom_s"][:, :, 0].astype(np.float64)
    pts, vel, cnt = scan_to_points(torch.from_numpy(states), torch.from_numpy(ranges), scan, max_points=mp, velocity=torch.from_numpy(velocity))
    pan = make_pan(cfg, K=1, N=mp, max_envs=B)
    dev = pts.device
    t = lambda k: torch.from_numpy(inp[k]).to(dev)
    S, U, D = pan(t("nom_s"), t("nom_u"), t("ref_s"), t("ref_us"), pts, vel, cnt)
    o_pts, o_vel, o_cnt = oscan.scan_batch(states, ranges, scan, max_points=mp, velocity=velocity)
    assert np.array_equal(o_cnt, cnt.cpu().numpy()) and (o_cnt == mp).all()
    pan2 = make_pan(cfg, K=1, N=mp, max_envs=B)
    S2, U2, D2 = pan2(t("nom_s"), t("nom_u"), t("ref_s"), t("ref_us"), torch.from_numpy(o_pts).to(dev), torch.from_numpy(o_vel).to(dev))
    assert torch.allclose(S, S2, atol=1e-4) and torch.allclose(U, U2, atol=1e-4)


@pytest.mark.gpu
def test_scan_argument_errors():
    import torch

    from neupan_b200 import scan_to_points

    scan = dict(angle_min=-1.0, angle_max=1.0, range_min=0.1, range_max=5.0)
    with pytest.raises(ValueError):
        scan_to_points(torch.zeros(2, 3), torch.ones(2, 16), scan, down_sample=0)
    with pytest.raises(ValueError):
        scan_to_points(torch.zeros(2, 3), torch.ones(2, 16), scan, velocity=torch.zeros(2, 2, 15))
