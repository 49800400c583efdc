"""Per-step InitialPath work (SURVEY 8f "next" row 1): oracle vs the reference class' golden vectors (CPU), batched CUDA
kernel vs both (GPU)."""
import importlib.util
import os

import numpy as np
import pytest

from oracle import ipath as oip

HERE = os.path.dirname(os.path.abspath(__file__))
_spec = importlib.util.spec_from_file_location("make_golden_ipath", os.path.join(HERE, "golden", "make_golden_ipath.py"))
mgi = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(mgi)
GOLD = np.load(os.path.join(HERE, "golden", "ref_ipath.npz"))
SC = mgi.SCENARIOS
T, DT, REF_SPEED = mgi.T, mgi.DT, mgi.REF_SPEED


def _gold(name):
    return {k.split(".", 1)[1]: GOLD[k] for k in GOLD.files if k.startswith(name + ".")}


def _oracle_for(name):
    kin, L, loop, step, split, curve, n = SC[name]
    o = oip.OracleInitialPath(T, DT, kin, L, loop)
    o.set_initial_path([p.copy() for p in mgi.make_path(n, step, split, curve)])
    return o


@pytest.mark.parametrize("name", list(SC))
def test_oracle_reproduces_reference_golden_vectors(name):
    """oracle/ipath.py replayed on the recorded inputs == what the reference class returned, bit for bit, including the
    headings the reference rewrote inside its stored path."""
    g, o = _gold(name), _oracle_for(name)
    for k in range(len(g["arrived"])):
        state = g["states"][k].reshape(3, 1)
        arrived = o.check_arrive(state)
        assert arrived == bool(g["arrived"][k]) and o.point_index == g["point_index"][k] and o.curve_index == g["curve_index"][k]
        if arrived:
            break
        nom_s, nom_u, ref_s, ref_us = o.generate_nom_ref_state(state, g["vel"][k], REF_SPEED)
        assert np.array_equal(nom_s, g["nom_s"][k]) and np.array_equal(ref_s, g["ref_s"][k]) and np.array_equal(ref_us, g["ref_us"][k])
    assert np.array_equal(np.hstack([p for c in o.curve_list for p in c]).T, g["final_path"])


class _RecordedReference:
    """The reference's InitialPath replayed from its recorded answers (ref_calls.npz): every call must arrive with the
    state and velocities it was recorded with."""

    def __init__(self, z):
        self.z, self.k, self.answered = z, 0, 0

    def set_initial_path(self, path):
        pass

    def check_arrive(self, state):
        assert np.array_equal(state, self.z["ipath.states"][self.k])
        self.point_index, self.curve_index = self.z["ipath.point_index"][self.k], self.z["ipath.curve_index"][self.k]
        self.k += 1
        return bool(self.z["ipath.arrived"][self.k - 1])

    def generate_nom_ref_state(self, state, vel, ref_speed):
        assert np.array_equal(vel, self.z["ipath.vel"][self.k - 1]) and ref_speed == REF_SPEED
        j, self.answered = self.answered, self.answered + 1
        return tuple(self.z[f"ipath.{key}"][j].copy() for key in ("nom_s", "nom_u", "ref_s", "ref_us"))


def test_golden_vectors_are_current():
    kin, L, loop, step, split, curve, n = SC["acker_two_gears"]
    ip, rows = _RecordedReference(np.load(os.path.join(HERE, "golden", "ref_calls.npz"))), []
    mgi.drive(ip, mgi.make_path(n, step, split, curve), 500 + list(SC).index("acker_two_gears"),
              lambda k, s, v, a, o, pi, ci: rows.append((a, None if o is None else o[2].copy())))
    g = _gold("acker_two_gears")
    assert len(rows) == len(g["arrived"]) == ip.k
    for k, (a, ref_s) in enumerate(rows):
        assert a == bool(g["arrived"][k]) and (a or np.array_equal(ref_s, g["ref_s"][k]))


def test_the_reference_rewrites_its_path_and_the_oracle_follows():
    """the view semantics are real: after a run the stored headings differ from the path that was set"""
    name = "acker_two_gears"
    kin, L, loop, step, split, curve, n = SC[name]
    before = np.hstack(mgi.make_path(n, step, split, curve)).T
    after = _gold(name)["final_path"]
    assert np.array_equal(before[:, [0, 1, 3]], after[:, [0, 1, 3]]) and not np.array_equal(before[:, 2], after[:, 2])


@pytest.mark.parametrize("name", list(SC))
def test_host_initial_path_of_the_facade_reproduces_the_reference(name):
    """neupan_b200.blocks.InitialPath (the single-robot host class behind the `neupan` facade) replayed on the recorded inputs:
    bit for bit what the reference class returned, including the path it leaves behind."""
    from neupan_b200.blocks.initial_path import InitialPath

    kin, L, loop, step, split, curve, n = SC[name]
    rb = type("Robot", (), dict(kinematics=kin, L=L, max_speed=np.array([8.0, 1.0])))()
    ip = InitialPath(T, DT, REF_SPEED, rb, loop=loop)
    ip.set_initial_path([p.copy() for p in mgi.make_path(n, step, split, curve)])
    g = _gold(name)
    for k in range(len(g["arrived"])):
        state = g["states"][k].reshape(3, 1)
        arrived = ip.check_arrive(state)
        assert arrived == bool(g["arrived"][k]) and ip.point_index == g["point_index"][k] and ip.curve_index == g["curve_index"][k]
        if arrived:
            break
        nom_s, nom_u, ref_s, ref_us = ip.generate_nom_ref_state(state, g["vel"][k], REF_SPEED)
        assert np.array_equal(nom_s, g["nom_s"][k]) and np.array_equal(ref_s, g["ref_s"][k]) and np.array_equal(np.asarray(ref_us), g["ref_us"][k])
    assert np.array_equal(np.hstack([p for c in ip.curve_list for p in c]).T, g["final_path"])


def test_pack_paths_layout():
    paths = [mgi.make_path(12, 0.4, 5, 0.0), mgi.make_path(7, 0.4, None, 0.0)]
    pts, cb, eb = oip.pack_paths(paths)
    assert pts.shape == (19, 4) and list(cb) == [0, 5, 12, 19] and list(eb) == [0, 2, 3]


# ---------------------------------------------------------------------------------------------------
def _ulp_close(a, w):
    w32 = np.asarray(w, np.float64).astype(np.float32)
    return np.all(np.abs(np.asarray(a, np.float32) - w32) <= np.spacing(np.maximum(np.abs(w32), np.float32(1e-30))))


@pytest.mark.gpu
@pytest.mark.parametrize("group", ["diff", "acker", "omni", "diff_loop", "acker_loop"])
def test_kernel_follows_the_reference_golden_runs(group):
    """nb_ipath_step through the C ABI: several recorded runs stepped in lockstep as one batch.  Indices, arrive flags and
    ref_us are exact; trajectories within 1 float32 ulp of the float32 cast of the reference's float64 values (FP64 cos / sin /
    tan of CUDA vs libm); the mutated path the handle holds equals the path the reference was left with (1e-12)."""
    import torch

    from neupan_b200 import InitialPathBatch

    names = [n for n in SC if (SC[n][0] + ("_loop" if SC[n][2] else "")) == group]
    kin, L, loop = SC[names[0]][0], SC[names[0]][1], SC[names[0]][2]
    golds = [_gold(n) for n in names]
    paths = [mgi.make_path(SC[n][6], SC[n][3], SC[n][4], SC[n][5]) for n in names]
    ipb = InitialPathBatch(T, DT, kin, L, loop, max_envs=len(names))
    ipb.set_initial_paths(paths)
    steps = max(len(g["arrived"]) for g in golds)
    for k in range(steps):
        idx = [min(k, len(g["arrived"]) - 1) for g in golds]  # a finished run keeps presenting its last state
        states = np.stack([g["states"][i] for g, i in zip(golds, idx)])
        vel = np.stack([g["vel"][i] for g, i in zip(golds, idx)])
        nom_s, nom_u, ref_s, ref_us, arrived = (x.cpu().numpy() for x in ipb.step(torch.from_numpy(states), torch.from_numpy(vel), REF_SPEED))
        st = ipb.read_state()
        for e, (g, i) in enumerate(zip(golds, idx)):
            if k >= len(g["arrived"]):
                assert arrived[e] == 1  # stays arrived
                continue
            assert bool(arrived[e]) == bool(g["arrived"][i]), (names[e], k)
            assert st["point_index"][e].item() == g["point_index"][i] and st["curve_index"][e].item() == g["curve_index"][i], (names[e], k)
            if arrived[e]:
                continue
            assert np.array_equal(nom_u[e], vel[e].astype(np.float32))
            assert np.array_equal(ref_us[e], g["ref_us"][i].astype(np.float32)), (names[e], k)
            assert _ulp_close(nom_s[e], g["nom_s"][i]), (names[e], k, np.abs(nom_s[e] - g["nom_s"][i]).max())
            assert _ulp_close(ref_s[e], g["ref_s"][i]), (names[e], k, np.abs(ref_s[e] - g["ref_s"][i]).max())
    final = ipb.read_state()["points"]
    want = np.vstack([g["final_path"] for g in golds])
    arrived_runs = [bool(g["arrived"][-1]) for g in golds]
    o = 0
    for g, done in zip(golds, arrived_runs):
        n = g["final_path"].shape[0]
        if done or len(g["arrived"]) == steps:  # runs that ended earlier than the batch kept stepping: only the others compare
            assert np.abs(final[o:o + n] - g["final_path"]).max() < 1e-12
        o += n
    assert want.shape == final.shape
    ipb.close()


@pytest.mark.gpu
def test_kernel_outputs_drive_pan_forward():
    """InitialPathBatch.step -> PAN.forward on the device, against the host InitialPath of the facade per environment."""
    import dataclasses

    import torch

    from gpu_helpers import make_pan
    from helpers import CONFIGS, make_inputs
    from neupan_b200 import InitialPathBatch

    cfg = dataclasses.replace(CONFIGS["C4"], K=1)
    B = 6
    inp = make_inputs(cfg, B=B, N=64)
    paths = [mgi.make_path(40, 0.4 + 0.0001 * (b - 3), None, 0.02 * (b - 2)) for b in range(B)]
    ipb = InitialPathBatch(cfg.T, cfg.dt, "diff", max_envs=B)
    ipb.set_initial_paths(paths)
    states = np.tile(np.array([0.05, -0.03, 0.25]), (B, 1))
    vel = np.zeros((B, 2, cfg.T), np.float32)
    vel[:, 0] = 3.0
    nom_s, nom_u, ref_s, ref_us, arrived = ipb.step(torch.from_numpy(states), torch.from_numpy(vel), 4.0)
    assert (arrived == 0).all()
    pan = make_pan(cfg, K=1, N=64, max_envs=B)
    t = lambda a: torch.from_numpy(a).cuda()
    S, U, D = pan(nom_s, nom_u, ref_s, ref_us, t(inp["points"]), t(inp["velocities"]))
    assert torch.isfinite(S).all() and (pan.status == 0).all()
    for b in range(B):  # the same step with the oracle, then PAN on its (float32) trajectories
        o = oip.OracleInitialPath(cfg.T, cfg.dt, "diff")
        o.set_initial_path([p.copy() for p in paths[b]])
        assert o.check_arrive(states[b].reshape(3, 1)) is False
        ns, nu, rs, ru = o.generate_nom_ref_state(states[b].reshape(3, 1), vel[b].astype(np.float64), 4.0)
        assert _ulp_close(nom_s[b].cpu().numpy(), ns) and _ulp_close(ref_s[b].cpu().numpy(), rs)
    ipb.close()


@pytest.mark.gpu
def test_ipath_argument_errors():
    import torch

    from neupan_b200 import InitialPathBatch

    with pytest.raises(ValueError):
        InitialPathBatch(10, 0.1, "tricycle")
    with pytest.raises(ValueError):
        InitialPathBatch(10, 0.1, "acker", wheelbase=None)
    ipb = InitialPathBatch(10, 0.1, "diff", max_envs=2)
    with pytest.raises(ValueError):
        ipb.step(torch.zeros(0, 3), torch.zeros(0, 2, 10), 4.0)  # no path set
    with pytest.raises(ValueError):
        ipb.set_initial_paths([mgi.make_path(5, 0.4, None, 0.0)] * 3)  # above max_envs
    ipb.close()
