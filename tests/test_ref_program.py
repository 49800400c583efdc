"""Pins the NRMP convex program to the REFERENCE'S OWN CODE (VERDICT r1, weak #1 / next #2).

``oracle/cvx_shim.py`` stands in for cvxpy / cvxpylayers, so ``neupan/blocks/nrmp.py:263-383`` and
``neupan/robot/robot.py:73-236`` execute unmodified and produce the program as arrays; ``tests/golden/ref_calls.npz``
holds those arrays and what the reference returned (made by ``tests/golden/make_golden_refcalls.py``).  Checked here, for
diff / acker / omni, scalar and vector q_s, with and without obstacle rows:

* the reference's objective equals ``oracle.nrmp.objective`` at random points (feasible or not);
* the oracle's optimum (float64 interior point, ``oracle/ipm.py``) satisfies the reference's constraints and passes a
  solver-free KKT certificate *of the reference's program*;
* the reference's own ``NRMP.forward`` (shim solver: HiGHS + active-set polish) returned the same trajectory;
* the reference's whole ``PAN.forward`` (its torch DUNE code + its NRMP through the shim) agrees with ``oracle.pan.OraclePAN``.

What stays unobservable: ECOS' own output.
"""
import importlib.util
import os

import numpy as np
import pytest

from helpers import GOLDEN, CONFIGS, make_inputs, oracle_factory, robot_spec
from oracle import dune as od, ipm as oipm, nrmp as onr

_spec = importlib.util.spec_from_file_location("make_golden_refcalls", os.path.join(GOLDEN, "make_golden_refcalls.py"))
mgr = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(mgr)
GOLD = np.load(os.path.join(GOLDEN, "ref_calls.npz"))
CASES = mgr.CASES


def _problem_and_reference(cname, adjust_over, M, scene="obstacles", env=0):
    """(cfg, the reference's program, the oracle's program, the reference's float64 solution, its (S, U, D)) of a case."""
    cfg, adjust, Mv, inp = mgr.program_inputs(cname, adjust_over, M, scene, env)
    i = CASES.index((cname, adjust_over, M))
    can = mgr.canonical_from(GOLD, f"program.{i}")
    if Mv > 0:
        mu, lam, sp, h, spec = mgr.dune_lists(cfg, inp)
        fa, fb = od.nrmp_coefficients(h, mu, lam, sp, cfg.T, Mv)
        fa, fb = fa.numpy(), fb.numpy()
    else:
        _, spec = robot_spec(cfg)
        fa = fb = None
    adj = onr.Adjust(**adjust)
    prob = onr.build_problem(spec, adj, inp["nom_s"][0], inp["nom_u"][0], inp["ref_s"][0], inp["ref_us"][0], fa, fb, Mv)
    ref = (GOLD[f"program.{i}.S"], GOLD[f"program.{i}.U"], GOLD[f"program.{i}.D"] if Mv > 0 else None)
    return cfg, can, prob, GOLD[f"program.{i}.x"], ref


def _stack_x(prob, S, U, D):
    parts = [np.asarray(S, float).reshape(-1), np.asarray(U, float).reshape(-1)]
    if prob.M > 0:
        parts.append(np.asarray(D, float).reshape(-1))
    return np.concatenate(parts)


@pytest.mark.parametrize("cname,adjust,M", CASES)
def test_reference_objective_equals_oracle_objective(cname, adjust, M):
    cfg, can, prob, _, _ = _problem_and_reference(cname, adjust, M)
    rng = np.random.default_rng(5)
    for _ in range(6):
        S = prob.nom_s + rng.normal(0, 0.5, prob.nom_s.shape)
        U = rng.normal(0, 2.0, (2, prob.T))
        D = rng.uniform(-0.5, 1.5, (1, prob.T))
        a, b = can.objective(_stack_x(prob, S, U, D)), onr.objective(prob, S, U, D[0])
        assert abs(a - b) <= 1e-9 * max(1.0, abs(b)), (a, b)


@pytest.mark.parametrize("cname,adjust,M", CASES)
def test_oracle_optimum_is_optimal_for_the_reference_program(cname, adjust, M):
    cfg, can, prob, xr, (Sr, Ur, Dr) = _problem_and_reference(cname, adjust, M)
    S, U, D, _ = oipm.solve_ipm(prob)
    x = _stack_x(prob, S, U, D)
    res, viol = can.kkt_certificate(x, act_tol=1e-7)
    scale = max(1.0, float(np.abs(can.gradient(x)).max()))
    assert viol < 1e-8, viol  # the reference's constraints hold at the oracle's optimum
    assert res < 2e-6 * scale, (res, scale)  # and its gradient is a combination of active normals
    # the reference's own forward (shim solver) lands on the same point; xr: float64, before its cast to float32 (nrmp.py:145-148)
    assert can.violation(xr) < 1e-8
    assert can.objective(x) <= can.objective(xr) + 1e-8 * max(1.0, abs(can.objective(xr)))
    assert np.abs(U - Ur).max() < 2e-5 and np.abs(S - Sr).max() < 2e-5
    if prob.M > 0:
        assert np.abs(D - Dr).max() < 2e-5


def test_reference_parameter_values_equal_oracle_parameters():
    """generate_parameter_value of the reference (nrmp.py:152-166, robot.py:239-316) vs oracle.nrmp.build_problem: bit for bit."""
    for cname in mgr.PARAM_CONFIGS:
        cfg, _, prob, _, _ = _problem_and_reference(cname, {}, None)
        vals = [GOLD[f"params.{cname}.{k}"] for k in range(int(GOLD[f"params.{cname}"]))]
        T = cfg.T
        assert np.array_equal(vals[0], prob.nom_s.astype(np.float32))
        assert np.array_equal(vals[1], prob.gamma_a.astype(np.float32))
        assert np.array_equal(vals[2], prob.gamma_b.astype(np.float32))
        for k in range(T):
            assert np.array_equal(vals[3 + k], prob.A[k].astype(np.float32))
            assert np.array_equal(vals[3 + T + k], prob.B[k].astype(np.float32))
            assert np.array_equal(vals[3 + 2 * T + k].reshape(-1), prob.C[k].astype(np.float32))
            assert np.array_equal(vals[3 + 3 * T + k], prob.fa[k].astype(np.float32))
            assert np.array_equal(vals[3 + 4 * T + k].reshape(-1), prob.fb[k].astype(np.float32))


@pytest.mark.parametrize("cname,K", [("C1", 2), ("C2", 3), ("C5", 2)])
def test_reference_pan_forward_equals_oracle_pan(cname, K):
    """The reference's PAN.forward end to end (pan.py:109-147) with only the solver swapped vs OraclePAN."""
    cfg = CONFIGS[cname]
    N = min(cfg.N, 150)
    inp = make_inputs(cfg, B=2, N=N, scene="obstacles")
    for b in range(2):
        g = f"pan.{cname}.{K}.{b}"
        S, U, D = GOLD[f"{g}.S"], GOLD[f"{g}.U"], GOLD[f"{g}.D"]
        op_ = oracle_factory(cfg, K=K, N=N)()
        vel = None if inp["velocities"] is None else inp["velocities"][b]
        So, Uo, Do = op_.forward(inp["nom_s"][b], inp["nom_u"][b], inp["ref_s"][b], inp["ref_us"][b], inp["points"][b], vel)
        assert np.abs(S - So).max() < 1e-4 and np.abs(U - Uo).max() < 1e-4 and np.abs(D - Do).max() < 1e-4
        assert abs(float(GOLD[f"{g}.min_distance"]) - op_.min_distance) < 1e-6
