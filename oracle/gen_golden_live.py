"""TEST INFRASTRUCTURE ONLY.  tests/golden/reference_live.npz + reference_live_shapes.json: what the tests of
tests/test_oracle.py that once ran the UNMODIFIED reference at test time compared against, recorded once so that they
run anywhere.

    python -m oracle.gen_golden_live       # from the repo root; needs /root/reference

  * `live_<case>`: the reference's energies on the spherenet_qm9 / dimenetpp_md17 case fixtures' inputs and weights,
    from a run of its own (a check on the case fixtures as well as on the restatement);
  * `nodefeat<i>_*`: SphereNet's node-feature options (spherenet.py:54-91,259-267), inputs + the reference's energies,
    with the state_dict shapes of both models in the JSON file;
  * `gsn_*`: inputs and outputs of ggraph3D/method/G_SphereNet/model/geometric_computing.py:xyztodat;
  * `ckpt_*`: a seeded sample of the shipped IS2RE checkpoint of ComENet-OCP (16.7 MB, too large to store): every value of
    `module.emb.emb.weight` and 16 (flat index, value) pairs of every other tensor.
"""
import importlib.util
import json
import os
import sys
import warnings

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import FIXTURE_THREADS, restated, shim  # noqa: E402
from oracle.gen_golden import CASES  # noqa: E402
from oracle.ocp_stub import OCP_DIR  # noqa: E402
from oracle.ref_loader import REFERENCE_ROOT, load_reference  # noqa: E402
from oracle.weights import formula_state_dict  # noqa: E402
from dig_b200.data import Batch, synthetic_batch  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
warnings.filterwarnings("ignore")

LIVE_CASES = ("spherenet_qm9", "dimenetpp_md17")
NODE_FEATURE_KW = (dict(use_node_features=False), dict(use_extra_node_feature=True, extra_node_feature_dim=3))
CKPT_SAMPLES = 16


def _np(t):
    return t.detach().cpu().numpy()


def main():
    torch.set_num_threads(FIXTURE_THREADS)
    method = load_reference()
    out, shapes = {}, {}
    for name in LIVE_CASES:
        g = np.load(os.path.join(GOLD, name + ".npz"))
        model_name, kw, _, wseed = CASES[name]
        model = getattr(method, model_name)(**kw)
        model.load_state_dict(formula_state_dict(model.state_dict(), seed=wseed))
        with torch.no_grad():
            e = model(Batch(z=torch.from_numpy(g["z"]), pos=torch.from_numpy(g["pos"]), batch=torch.from_numpy(g["batch"])))
        out["live_" + name] = _np(e)

    for i, kw in enumerate(NODE_FEATURE_KW):
        torch.manual_seed(0)
        model = method.SphereNet(cutoff=5.0, num_layers=2, **kw)
        model.load_state_dict(formula_state_dict(model.state_dict(), seed=11))
        shapes["SphereNet" + json.dumps(dict(cutoff=5.0, num_layers=2, **kw), sort_keys=True)] = \
            {k: list(v.shape) for k, v in model.state_dict().items()}
        b = synthetic_batch(3, "qm9", seed=6)
        nf = torch.randn(b.z.numel(), 3) if "extra_node_feature_dim" in kw else None
        with torch.no_grad():
            e = model(Batch(z=b.z, pos=b.pos, batch=b.batch, node_feature=nf))
        out.update({f"nodefeat{i}_z": _np(b.z), f"nodefeat{i}_pos": _np(b.pos), f"nodefeat{i}_batch": _np(b.batch),
                    f"nodefeat{i}_energy": _np(e)})
        if nf is not None:
            out[f"nodefeat{i}_node_feature"] = _np(nf)

    shim.install()
    path = os.path.join(REFERENCE_ROOT, "dig", "ggraph3D", "method", "G_SphereNet", "model", "geometric_computing.py")
    spec = importlib.util.spec_from_file_location("gsn_geo", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    b = synthetic_batch(5, "qm9", seed=9, variable=True)
    ei = restated.radius_graph(b.pos, 5.0, b.batch)
    want = mod.xyztodat(b.pos, ei, b.pos.size(0), b.batch)
    out.update({"gsn_pos": _np(b.pos), "gsn_batch": _np(b.batch), "gsn_edge_index": _np(ei),
                "gsn_n_out": np.int64(len(want))})
    out.update({f"gsn_out{k}": _np(w) for k, w in enumerate(want)})

    ck = torch.load(os.path.join(OCP_DIR, "IS2RETrainedModelWeights.pt"), map_location="cpu", weights_only=False)
    sd = ck["state_dict"]
    gen = torch.Generator().manual_seed(0)
    keys = sorted(sd)
    idx, val, owner = [], [], []
    for n, k in enumerate(keys):
        flat = sd[k].reshape(-1)
        take = torch.randperm(flat.numel(), generator=gen)[:CKPT_SAMPLES]
        idx.append(take)
        val.append(flat[take].float())
        owner.append(torch.full_like(take, n))
    out.update({"ckpt_keys": np.array(keys), "ckpt_owner": _np(torch.cat(owner)), "ckpt_index": _np(torch.cat(idx)),
                "ckpt_value": _np(torch.cat(val)), "ckpt_emb_weight": _np(sd["module.emb.emb.weight"].float())})

    np.savez_compressed(os.path.join(GOLD, "reference_live.npz"), **out)
    with open(os.path.join(GOLD, "reference_live_shapes.json"), "w") as fh:
        json.dump(shapes, fh)
    print("reference_live:", {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
