"""Golden vectors for the tests that compare with the reference's own code directly, recorded from that code so that the
tests run without it:

* ``program.*`` -- for every case of ``CASES``: the NRMP program the reference's ``nrmp.py`` / ``robot.py`` build, as the
  arrays ``oracle/cvx_shim.py`` turns it into, and what its ``NRMP.forward`` returns (the shim solver's float64 point and the
  cast trajectories); ``params.*`` -- its ``generate_parameter_value``; ``pan.*`` -- its whole ``PAN.forward``
  (``tests/test_ref_program.py``);
* ``dune.*`` -- its ``DUNE.forward`` on the acker checkpoint and the checkpoint's digest (``tests/test_oracle_dune.py``);
* ``scan.*`` -- the calls its ``scan_to_point_velocity`` answered for the ``velocity_stride`` case of ``ref_scan.npz``
  (``tests/test_scan.py``);
* ``ipath.*`` -- the calls its ``InitialPath`` answered in the ``acker_two_gears`` run of ``ref_ipath.npz``
  (``tests/test_ipath.py``).

    python tests/golden/make_golden_refcalls.py     # needs the reference checkout (oracle/refload.py); writes tests/golden/ref_calls.npz
"""
import hashlib
import importlib.util
import os
import sys
import tempfile
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for _p in (ROOT, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from helpers import CONFIGS, make_inputs, robot_spec, weights_path  # noqa: E402
from oracle import cvx_shim, dune as od  # noqa: E402

OUT = os.path.join(HERE, "ref_calls.npz")

# (config, adjust overrides, nrmp_max_num override or None)
CASES = [("C1", {}, None), ("C2", {}, None), ("C4", {}, None), ("C5", {}, None),
         ("C4", dict(q_s=[0.5, 1.5, 0.25]), None), ("C2", dict(q_s=[1.0, 0.3, 2.0], p_u=0.7, eta=8.0, d_max=1.5, d_min=0.2), None),
         ("C1", {}, 0), ("C5", dict(q_s=[1.0, 2.0, 3.0]), 0)]
PARAM_CONFIGS = ("C1", "C2", "C5")
PAN_CASES = [("C1", 2), ("C2", 3), ("C5", 2)]
DUNE_CHECKPOINT = "example/model/acker_robot_default/model_5000.pth"


def program_inputs(cname, adjust_over, M, scene="obstacles", env=0):
    """(cfg, adjust, M, inputs of one environment) of a program case."""
    cfg = CONFIGS[cname]
    adjust = dict(cfg.adjust); adjust.update(adjust_over)
    inp = make_inputs(cfg, B=1, N=min(cfg.N, 120), scene=scene, env_offset=env)
    return cfg, adjust, cfg.M if M is None else M, inp


def dune_lists(cfg, inp, b=0):
    """mu / lam / sorted point lists of one environment from the (reference-pinned) DUNE oracle."""
    rb, spec = robot_spec(cfg)
    w = od.load_weights(weights_path(cfg.model))
    G, h = torch.from_numpy(spec.G).float(), torch.from_numpy(spec.h.reshape(-1, 1)).float()
    t = lambda a: None if a is None else torch.from_numpy(a[b])
    vel = None if inp["velocities"] is None else t(inp["velocities"])
    p0, R, p = od.point_flow(t(inp["nom_s"]), t(inp["points"]), vel, cfg.T, cfg.dt, cfg.N)
    mu, lam, sp, _, _ = od.dune_forward(w, G, h, p0, R, p)
    return mu, lam, sp, h, spec


def weights_digest(w) -> str:
    h = hashlib.sha256()
    for k in sorted(w):
        h.update(k.encode()); h.update(np.ascontiguousarray(w[k].numpy(), np.float32).tobytes())
    return h.hexdigest()


def canonical_arrays(can, prefix):
    """cvx_shim.Canonical -> flat {key: array} (inverse: canonical_from)."""
    assert not can.soc
    out = {f"{prefix}.{k}": np.asarray(getattr(can, k)) for k in ("n", "l", "const", "E", "e", "G", "g", "lb")}
    for kind in ("quads", "hinges"):
        terms = getattr(can, kind)
        out[f"{prefix}.{kind}"] = np.array(len(terms))
        for j, (c, a) in enumerate(terms):
            out[f"{prefix}.{kind}.{j}.c"], out[f"{prefix}.{kind}.{j}.A"] = np.asarray(c, float), a.A
            out[f"{prefix}.{kind}.{j}.b"], out[f"{prefix}.{kind}.{j}.shape"] = a.b, np.asarray(a.shape, np.int64)
    return out


def canonical_from(z, prefix):
    terms = {kind: [(float(z[f"{prefix}.{kind}.{j}.c"]), cvx_shim._Aff(z[f"{prefix}.{kind}.{j}.A"], z[f"{prefix}.{kind}.{j}.b"], tuple(z[f"{prefix}.{kind}.{j}.shape"])))
                    for j in range(int(z[f"{prefix}.{kind}"]))] for kind in ("quads", "hinges")}
    return cvx_shim.Canonical(int(z[f"{prefix}.n"]), terms["quads"], terms["hinges"], z[f"{prefix}.l"], float(z[f"{prefix}.const"]),
                              z[f"{prefix}.E"], z[f"{prefix}.e"], z[f"{prefix}.G"], z[f"{prefix}.g"], [], z[f"{prefix}.lb"])


def _load_fixture_module(name):
    spec = importlib.util.spec_from_file_location(name, os.path.join(HERE, f"{name}.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


# ------------------------------------------------------------------------------------------------------------------
def _program(out):
    from neupan.blocks.nrmp import NRMP
    from neupan.blocks.pan import PAN as RefPAN
    from neupan.robot import robot as RefRobot

    t = lambda a: torch.from_numpy(a[0])
    layers = {}
    for i, (cname, adjust_over, M) in enumerate(CASES):
        cfg, adjust, Mv, inp = program_inputs(cname, adjust_over, M)
        layer = NRMP(cfg.T, cfg.dt, RefRobot(cfg.T, cfg.dt, **cfg.robot_kwargs), nrmp_max_num=Mv, **adjust)
        args = [t(inp["nom_s"]), t(inp["nom_u"]), t(inp["ref_s"]), t(inp["ref_us"])]
        if Mv > 0:
            args += list(dune_lists(cfg, inp)[:3])
        S, U, D = layer.forward(*args)
        out.update(canonical_arrays(layer.nrmp_layer.last_canonical, f"program.{i}"))
        out[f"program.{i}.x"] = layer.nrmp_layer.last_x
        out[f"program.{i}.S"], out[f"program.{i}.U"] = S.numpy(), U.numpy()
        if Mv > 0:
            out[f"program.{i}.D"] = D.numpy()
        if not adjust_over and M is None:
            layers[cname] = (layer, args)
    for cname in PARAM_CONFIGS:
        layer, args = layers[cname]
        for k, v in enumerate(layer.generate_parameter_value(*args)):
            out[f"params.{cname}.{k}"] = v.detach().numpy()
        out[f"params.{cname}"] = np.array(k + 1)

    with tempfile.TemporaryDirectory() as tmp:
        for cname, K in PAN_CASES:
            cfg = CONFIGS[cname]
            N = min(cfg.N, 150)
            inp = make_inputs(cfg, B=2, N=N, scene="obstacles")
            ck = os.path.join(tmp, f"{cfg.model}.pth")
            torch.save(dict(od.load_weights(weights_path(cfg.model))), ck)
            for b in range(2):
                rp = RefPAN(cfg.T, cfg.dt, RefRobot(cfg.T, cfg.dt, **cfg.robot_kwargs), iter_num=K, dune_max_num=N, nrmp_max_num=cfg.M,
                            dune_checkpoint=ck, iter_threshold=0.0, adjust_kwargs=dict(cfg.adjust))
                tb = lambda a: None if a is None else torch.from_numpy(a[b])
                S, U, D = rp(tb(inp["nom_s"]), tb(inp["nom_u"]), tb(inp["ref_s"]), tb(inp["ref_us"]), tb(inp["points"]), tb(inp["velocities"]))
                p = f"pan.{cname}.{K}.{b}"
                out[f"{p}.S"], out[f"{p}.U"], out[f"{p}.D"] = S.numpy(), U.numpy(), D.numpy()
                out[f"{p}.min_distance"] = np.asarray(float(rp.min_distance))


def _dune(out, reference_root):
    from neupan.blocks import DUNE, PAN
    from neupan.robot import robot as RefRobot

    rr = RefRobot(10, 0.1, kinematics="acker", length=4.6, width=1.6, wheelbase=3)
    ck = os.path.join(reference_root, DUNE_CHECKPOINT)
    dune = DUNE(10, ck, rr, 80, {})
    fake = types.SimpleNamespace(T=10, dt=0.1, dune_max_num=80, printed=True, print_once=lambda *_: None)
    fake.point_state_transform = types.MethodType(PAN.point_state_transform, fake)
    g = torch.Generator().manual_seed(3)
    nom_s = torch.randn(3, 11, generator=g); pts = 6 * torch.randn(2, 200, generator=g); vel = torch.randn(2, 200, generator=g)
    pf, Rl, pl = PAN.generate_point_flow(fake, nom_s, pts, vel)
    mu, lam, sp = dune(pf, Rl, pl)
    out["dune.nom_s"], out["dune.points"], out["dune.velocities"] = nom_s.numpy(), pts.numpy(), vel.numpy()
    out["dune.G"], out["dune.h"] = np.asarray(rr.G, np.float32), np.asarray(rr.h, np.float32)
    out["dune.mu"], out["dune.lam"], out["dune.sorted_points"] = (torch.stack(x).numpy() for x in (mu, lam, sp))
    out["dune.min_distance"] = np.asarray(float(dune.min_distance), np.float32)
    out["dune.checkpoint_sha256"] = np.array(weights_digest(od.load_weights(ck)))


def _scan(out, ref):
    from oracle import scan as oscan

    mgs = _load_fixture_module("make_golden_scan")
    gold = np.load(os.path.join(HERE, "ref_scan.npz"))
    B, R, scan, off, ar, ds, mp, vm = mgs.CASES["velocity_stride"]
    g = {k: gold[f"velocity_stride.{k}"] for k in ("states", "ranges", "velocity")}
    calls = []

    def fn_v(st, sc, o, a, d):
        p, v = ref.neupan.scan_to_point_velocity(None, st, sc, o, a, d)
        calls.append((st, sc["ranges"], sc["velocity"], p, v))
        return p, v

    oscan.scan_batch(g["states"], g["ranges"], scan, off, ar, ds, mp, g["velocity"], True, fn_velocity=fn_v)
    for i, (st, rg, vi, p, v) in enumerate(calls):
        out[f"scan.{i}.state"], out[f"scan.{i}.ranges"], out[f"scan.{i}.velocity"] = np.asarray(st), np.asarray(rg), np.asarray(vi)
        out[f"scan.{i}.points"], out[f"scan.{i}.vel"] = np.asarray(p), np.asarray(v)
    out["scan.calls"] = np.array(len(calls))


def _ipath(out):
    mgi = _load_fixture_module("make_golden_ipath")
    name = "acker_two_gears"
    kin, L, loop, step, split, curve, n = mgi.SCENARIOS[name]
    ip, rows = mgi.reference_instance(kin, L, loop), []
    mgi.drive(ip, mgi.make_path(n, step, split, curve), 500 + list(mgi.SCENARIOS).index(name),
              lambda k, s, v, a, o, pi, ci: rows.append((s.copy(), v.copy(), a, o, pi, ci)))
    out["ipath.states"] = np.stack([r[0] for r in rows])
    out["ipath.vel"] = np.stack([r[1] for r in rows])
    out["ipath.arrived"] = np.array([r[2] for r in rows])
    out["ipath.point_index"], out["ipath.curve_index"] = np.array([r[4] for r in rows]), np.array([r[5] for r in rows])
    answered = [r[3] for r in rows if r[3] is not None]
    for j, key in enumerate(("nom_s", "nom_u", "ref_s", "ref_us")):
        out[f"ipath.{key}"] = np.stack([np.asarray(o[j], float) for o in answered])


def main():
    from oracle import refload

    ref = refload.load_reference()
    out = {}
    _program(out)
    _dune(out, refload.REFERENCE_ROOT)
    _scan(out, ref)
    _ipath(out)
    np.savez_compressed(OUT, **out)
    print(OUT, os.path.getsize(OUT), "bytes,", len(out), "arrays")


if __name__ == "__main__":
    main()
