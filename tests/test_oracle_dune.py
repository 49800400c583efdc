"""Pins oracle/dune.py (the CPU restatement of the DUNE half) against the reference's own code:
golden vectors produced by that code (tests/golden/ref_dune_*.npz, made by make_golden.py, and
tests/golden/ref_calls.npz, made by make_golden_refcalls.py)."""
import numpy as np
import pytest
import torch

from helpers import GOLDEN, weights_path
from oracle import dune as od


@pytest.mark.parametrize("model", ["diff", "acker", "polygon"])
@pytest.mark.parametrize("case", ["a", "b", "c", "d"])
def test_dune_matches_reference_golden(model, case):
    z = np.load(f"{GOLDEN}/ref_dune_{model}.npz")
    w = od.load_weights(weights_path(model))
    G = torch.from_numpy(z["G"]).float(); h = torch.from_numpy(z["h"]).float()
    nom_s = torch.from_numpy(z[f"{case}_nom_s"]); pts = torch.from_numpy(z[f"{case}_points"])
    vel = z[f"{case}_vel"]; vel = None if vel.size == 0 else torch.from_numpy(vel)
    T = nom_s.shape[1] - 1
    p0, R, pl = od.point_flow(nom_s, pts, vel, T, 0.1, int(z[f"{case}_dune_max_num"]))
    mu, lam, sp, md, _ = od.dune_forward(w, G, h, p0, R, pl, stable=False)
    assert np.array_equal(torch.stack(p0).numpy(), z[f"{case}_p0"])
    assert np.array_equal(torch.stack(R).numpy(), z[f"{case}_R"])
    assert np.array_equal(torch.stack(mu).numpy(), z[f"{case}_mu"])  # bit-for-bit
    assert np.array_equal(torch.stack(lam).numpy(), z[f"{case}_lam"])
    assert np.array_equal(torch.stack(sp).numpy(), z[f"{case}_sorted_points"])
    assert np.float32(md) == z[f"{case}_min_distance"]
    assert np.array_equal(pl[0].numpy(), z[f"{case}_dune_points"])
    # the deterministic (stable) order differs from the reference order only inside exact ties
    mu_s, lam_s, sp_s, _, dist = od.dune_forward(w, G, h, p0, R, pl, stable=True)
    for t in range(T + 1):
        d_ref = od.objective_distance(G, h, mu[t], None if False else (R[t].T @ (sp[t] - nom_s[0:2, t:t + 1])))
        d_stb = od.objective_distance(G, h, mu_s[t], (R[t].T @ (sp_s[t] - nom_s[0:2, t:t + 1])))
        assert torch.equal(d_ref, d_stb)


def test_dune_matches_live_reference():
    """The reference's DUNE.forward on its acker checkpoint (recorded in ref_calls.npz) vs the oracle on the weights fixture."""
    import hashlib

    z = np.load(f"{GOLDEN}/ref_calls.npz")
    nom_s, pts, vel = (torch.from_numpy(z[f"dune.{k}"]) for k in ("nom_s", "points", "velocities"))
    w = od.load_weights(weights_path("acker"))
    p0, R, pl2 = od.point_flow(nom_s, pts, vel, 10, 0.1, 80)
    mu, lam, sp, md, _ = od.dune_forward(w, torch.from_numpy(z["dune.G"]), torch.from_numpy(z["dune.h"]), p0, R, pl2, stable=False)
    assert np.array_equal(torch.stack(mu).numpy(), z["dune.mu"])
    assert np.array_equal(torch.stack(lam).numpy(), z["dune.lam"])
    assert np.array_equal(torch.stack(sp).numpy(), z["dune.sorted_points"])
    assert np.float32(md) == z["dune.min_distance"]
    # weights fixture == checkpoint
    h = hashlib.sha256()
    for k in sorted(w):
        h.update(k.encode()); h.update(np.ascontiguousarray(w[k].numpy(), np.float32).tobytes())
    assert h.hexdigest() == str(z["dune.checkpoint_sha256"])
