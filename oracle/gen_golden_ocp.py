"""TEST INFRASTRUCTURE ONLY.  tests/golden/comenet_ocp.npz: the UNMODIFIED reference ComENet-OCP
(dig/threedgraph/method/comenet/ocp/comenet-ocp.py over oracle/shim.py + oracle/ocp_stub.py) on a synthetic periodic
batch, with formula weights; plus the key names / shapes of the shipped IS2RE checkpoint.

    python -m oracle.gen_golden_ocp        # from the repo root; needs /root/reference
"""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import FIXTURE_THREADS  # noqa: E402
from oracle.ocp_stub import OCP_DIR, load_comenet_ocp  # noqa: E402
from oracle.weights import formula_state_dict  # noqa: E402
from dig_b200.data import synthetic_pbc_batch  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
CTOR = dict(num_atoms=0, bond_feat_dim=0, hidden_channels=256, num_blocks=4, cutoff=6.0, num_radial=3,
            num_spherical=2, hetero=False, num_output_layers=3)          # ocp/comenet.yml
DATA = dict(nsys=3, natoms=30, seed=7)
WSEED = 21


def main():
    torch.set_num_threads(FIXTURE_THREADS)
    mod = load_comenet_ocp()
    torch.manual_seed(0)
    model = mod.ComENet(**CTOR)
    sd = formula_state_dict(model.state_dict(), seed=WSEED)
    sd["lin_out.weight"] = sd["lin_out.weight"] + 0.05          # the class initialises lin_out to zeros
    model.load_state_dict(sd)
    model.eval()
    b = synthetic_pbc_batch(**DATA)
    with torch.no_grad():
        e32 = model(b)
        m64 = model.double()
        b64 = synthetic_pbc_batch(**DATA)
        b64.pos, b64.cell = b64.pos.double(), b64.cell.double()
        e64 = m64(b64)
    np.savez(os.path.join(GOLD, "comenet_ocp.npz"), energy_f32=e32.numpy(), energy_f64=e64.numpy(),
             **{k: getattr(b, k).numpy() for k in ("atomic_numbers", "pos", "tags", "cell", "edge_index", "cell_offsets",
                                                   "neighbors", "batch")})
    ck = torch.load(os.path.join(OCP_DIR, "IS2RETrainedModelWeights.pt"), map_location="cpu", weights_only=False)
    shapes = {k: list(v.shape) for k, v in ck["state_dict"].items()}
    with open(os.path.join(GOLD, "comenet_ocp_checkpoint_shapes.json"), "w") as fh:
        json.dump({"keys": shapes, "num_params": int(sum(int(np.prod(s)) for s in shapes.values())),
                   "val_energy_mae": float(ck["val_metrics"]["energy_mae"]["metric"])
                   if isinstance(ck["val_metrics"].get("energy_mae"), dict) else None}, fh, indent=0)
    print("comenet_ocp: energies", e32.flatten().tolist(), "fp32-vs-fp64", float((e32 - e64.float()).abs().max() / e64.abs().max()))


if __name__ == "__main__":
    main()
