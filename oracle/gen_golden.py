"""TEST INFRASTRUCTURE ONLY.  Generates tests/golden/*.npz|json by running the UNMODIFIED
reference (/root/reference, over oracle/shim.py) in the build container.

    python -m oracle.gen_golden            # from the repo root; needs /root/reference

The reference cannot travel to the GPU box, so these fixtures (inputs + outputs; weights are
regenerated from key names by oracle/weights.py) are what `-m gpu` tests compare against.
All reference runs are CPU fp32 (and fp64 for the noise floor, SURVEY.md §5.9).
"""
import inspect
import json
import os
import sys
import warnings

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import FIXTURE_THREADS  # noqa: E402
from oracle.ref_loader import load_reference, load_reference_utils  # noqa: E402
from oracle.weights import formula_state_dict  # noqa: E402
from dig_b200.data import synthetic_batch, Batch  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
warnings.filterwarnings("ignore")

CASES = {
    # name: (model, ctor kwargs, data kwargs, weight seed)
    "schnet_cfg1": ("SchNet", dict(num_layers=2, hidden_channels=32, num_filters=32, cutoff=10.0),
                    dict(nmol=16, shape="schnet-plumbing", seed=0), 1),
    "spherenet_qm9": ("SphereNet", dict(cutoff=5.0), dict(nmol=6, shape="qm9", seed=2, variable=True), 2),
    "dimenetpp_md17": ("DimeNetPP", dict(cutoff=5.0), dict(nmol=4, shape="md17-aspirin", seed=3), 3),
    "comenet_oc20": ("ComENet", dict(cutoff=6.0, hidden_channels=256, middle_channels=64),
                     dict(nmol=2, shape="oc20-is2re", seed=4), 4),
    "spherenet_ns3": ("SphereNet", dict(cutoff=5.0, num_spherical=3),
                      dict(nmol=3, shape="qm9", seed=5), 5),
}


def _np(t):
    return t.detach().cpu().numpy()


def run_case(method, utils, name):
    model_name, ctor, data_kw, wseed = CASES[name]
    torch.manual_seed(0)
    model = getattr(method, model_name)(**ctor)
    sd = formula_state_dict(model.state_dict(), seed=wseed)
    model.load_state_dict(sd)
    model.eval()
    b = synthetic_batch(**data_kw)
    out = {"z": _np(b.z), "pos": _np(b.pos), "batch": _np(b.batch),
           "num_params": np.int64(sum(p.numel() for p in model.parameters()))}

    def fwd(dtype, want_force):
        m = model.to(dtype)
        pos = b.pos.to(dtype).clone().requires_grad_(want_force)
        bd = Batch(z=b.z, pos=pos, batch=b.batch)
        e = m(bd)
        f = None
        if want_force:
            f = -torch.autograd.grad(e.sum(), pos)[0]
        return e, f

    want_force = model_name in ("SchNet", "DimeNetPP")
    e32, f32 = fwd(torch.float32, want_force)
    out["energy_f32"] = _np(e32)
    if f32 is not None:
        out["force_f32"] = _np(f32)
    e64, f64 = fwd(torch.float64, want_force)
    out["energy_f64"] = _np(e64)
    if f64 is not None:
        out["force_f64"] = _np(f64)
    model.to(torch.float32)

    # graph + geometry intermediates (fp32)
    from oracle import shim
    cutoff = ctor.get("cutoff")
    ei = shim.radius_graph(b.pos, r=cutoff, batch=b.batch)
    out["edge_index"] = _np(ei)
    if model_name in ("SphereNet", "DimeNetPP"):
        tors = model_name == "SphereNet"
        res = utils.xyz_to_dat(b.pos, ei, b.z.size(0), use_torsion=tors)
        if tors:
            dist, angle, torsion, i, j, idx_kj, idx_ji = res
            out["torsion"] = _np(torsion)
        else:
            dist, angle, i, j, idx_kj, idx_ji = res
        out.update(dist=_np(dist), angle=_np(angle), idx_kj=_np(idx_kj), idx_ji=_np(idx_ji))
        emb = model.emb(dist, angle, torsion, idx_kj) if tors else model.emb(dist, angle, idx_kj)
        out["rbf0"] = _np(emb[0])
        out["sbf_head"] = _np(emb[1][:256])
        if tors:
            out["tbf_head"] = _np(emb[2][:64])
    elif model_name == "SchNet":
        row, col = ei
        out["dist"] = _np((b.pos[row] - b.pos[col]).norm(dim=-1))
    np.savez_compressed(os.path.join(GOLD, name + ".npz"), **out)
    print(name, "E", ei.size(1), "energy", out["energy_f32"].ravel()[:3],
          "max|f32-f64|/|f64|", float(np.abs(out["energy_f32"] - out["energy_f64"]).max()
                                    / np.abs(out["energy_f64"]).max()))


def basis_sources(method):
    """The lambdified source strings the reference builds for each (model, ns, nr)."""
    import dig.threedgraph.method.spherenet.features as fs
    import dig.threedgraph.method.dimenetpp.features as fd
    import dig.threedgraph.method.comenet.features as fc

    def src(f):
        s = inspect.getsource(f)
        return s.split("return", 1)[1].strip()

    def const0(fn):  # l = 0 closures are python lambdas around a constant
        v = fn(torch.zeros(1)) if fn.__code__.co_argcount == 1 else fn(torch.zeros(1), torch.zeros(1))
        return repr(float(v))

    out = {}
    for ns, nr in ((7, 6), (3, 6)):
        te = fs.torsion_emb(ns, nr)
        ae = fs.angle_emb(ns, nr)
        out[f"spherenet_{ns}_{nr}"] = {
            "bessel": [src(f) for f in te.bessel_funcs],
            "bessel_angle_emb": [src(f) for f in ae.bessel_funcs],
            "yl0": [const0(ae.sph_funcs[0])] + [src(f) for f in ae.sph_funcs[1:]],
            "ylm": [const0(te.sph_funcs[0])] + [src(f) for f in te.sph_funcs[1:]],
        }
    ad = fd.angle_emb(7, 6)
    out["dimenetpp_7_6"] = {
        "bessel": [src(f) for f in ad.bessel_funcs],
        "yl0": [const0(ad.sph_funcs[0])] + [src(f) for f in ad.sph_funcs[1:]],
    }
    tc = fc.torsion_emb(num_radial=3, num_spherical=2, cutoff=6.0)
    ac = fc.angle_emb(num_radial=3, num_spherical=2, cutoff=6.0)
    out["comenet_2_3"] = {
        "bessel": [src(f) for f in tc.bessel_funcs],
        "bessel_angle_emb": [src(f) for f in ac.bessel_funcs],
        "yl0": [const0(ac.sph_funcs[0])] + [src(f) for f in ac.sph_funcs[1:]],
        "ylm": [const0(tc.sph_funcs[0])] + [src(f) for f in tc.sph_funcs[1:]],
    }
    with open(os.path.join(GOLD, "basis_formulas.json"), "w") as fh:
        json.dump(out, fh, indent=1)
    print("basis formulas:", {k: {kk: len(vv) for kk, vv in v.items()} for k, v in out.items()})


def notebook_example(utils):
    """examples/threedgraph/xyz_to_dat.ipynb cells 4-6 (SURVEY.md §8c golden (1))."""
    ei = torch.tensor([[1, 0, 2, 1, 3, 2], [0, 1, 1, 2, 2, 3]])
    pos = torch.tensor([[0., 0, 0], [1, 1, 0], [2, 0, 0], [3, 1, 0]])
    dist, angle, torsion, i, j, idx_kj, idx_ji = utils.xyz_to_dat(pos, ei, 4, use_torsion=True)
    np.savez(os.path.join(GOLD, "xyz_to_dat_notebook.npz"), edge_index=_np(ei), pos=_np(pos),
             dist=_np(dist), angle=_np(angle), torsion=_np(torsion), idx_kj=_np(idx_kj), idx_ji=_np(idx_ji))
    print("notebook:", idx_kj.tolist(), idx_ji.tolist(), torsion.tolist())


def state_shapes(method):
    """Key names + shapes of every fixture model's state_dict (SURVEY.md Appendix A contract), so
    tests can rebuild formula weights and check the drop-in classes without the reference."""
    out = {}
    for name, (mn, kw, _, _) in CASES.items():
        model = getattr(method, mn)(**kw)
        out[mn + json.dumps(kw, sort_keys=True)] = {k: list(v.shape) for k, v in model.state_dict().items()}
    with open(os.path.join(GOLD, "state_shapes.json"), "w") as fh:
        json.dump(out, fh)
    print("state shapes:", {k: len(v) for k, v in out.items()})


def main():
    torch.set_num_threads(FIXTURE_THREADS)
    os.makedirs(GOLD, exist_ok=True)
    method = load_reference()
    utils = load_reference_utils()
    which = sys.argv[1:] or list(CASES) + ["basis", "notebook", "shapes"]
    for name in which:
        if name == "basis":
            basis_sources(method)
        elif name == "notebook":
            notebook_example(utils)
        elif name == "shapes":
            state_shapes(method)
        else:
            run_case(method, utils, name)


if __name__ == "__main__":
    main()
