"""CPU tests: the oracle against the reference's own known answers and against the golden fixtures.

* golden (1) examples/threedgraph/xyz_to_dat.ipynb: adj_t row-select, num_triplets, idx_kj/idx_ji
* golden (2) #Params: 1890118 for SphereNet(num_spherical=3)   (threedgraph.ipynb:173)
* golden (3) test/threedgraph/evaluation/test_ThreeDEvaluator.py:7-21 (MAE 0.45)
* oracle/restated.py == real reference, bit for bit, on every fixture case (CPU fp32)
"""
import json
import math
import os

import numpy as np
import pytest
import torch

from helpers import CASES, case_inputs, formula_state_dict, load_golden
from oracle import FIXTURE_THREADS, restated, shim


@pytest.fixture(autouse=True)
def _fixture_threads():
    """The bit-for-bit comparisons with the fixtures hold at the intra-op thread count they were written with."""
    n = torch.get_num_threads()
    torch.set_num_threads(FIXTURE_THREADS)
    yield
    torch.set_num_threads(n)


def test_notebook_sparse_tensor_known_answer():
    # examples/threedgraph/xyz_to_dat.ipynb cells 4-6
    ei = torch.tensor([[1, 0, 2, 1, 3, 2], [0, 1, 1, 2, 2, 3]])
    j, i = ei
    adj_t = shim.SparseTensor(row=i, col=j, value=torch.arange(6), sparse_sizes=(4, 4))
    sel = adj_t[j]
    assert sel.storage.row().tolist() == [0, 0, 1, 2, 2, 3, 3, 4, 5, 5]
    assert sel.storage.col().tolist() == [0, 2, 1, 1, 3, 0, 2, 2, 1, 3]
    assert sel.storage.value().tolist() == [1, 2, 0, 3, 4, 1, 2, 5, 3, 4]
    assert sel.set_value(None).sum(dim=1).to(torch.long).tolist() == [2, 1, 2, 2, 1, 2]


def test_notebook_xyz_to_dat_restated():
    g = load_golden("xyz_to_dat_notebook")
    pos = torch.from_numpy(g["pos"])
    ei = torch.from_numpy(g["edge_index"])
    dist, angle, torsion, i, j, idx_kj, idx_ji = restated.xyz_to_dat(pos, ei, 4, use_torsion=True)
    assert idx_kj.tolist() == [2, 4, 1, 3] and idx_ji.tolist() == [0, 2, 3, 5]
    assert torch.allclose(dist, torch.full((6,), math.sqrt(2.0)))
    assert torch.allclose(angle, torch.full((4,), math.pi / 2))
    assert np.array_equal(torsion.numpy(), g["torsion"])          # exactly 2*pi: integer coordinates


def test_scatter_min_semantics():
    src = torch.tensor([3.0, 1.0, 1.0, 5.0])
    idx = torch.tensor([0, 0, 0, 2])
    val, arg = shim.scatter_min(src, idx, dim_size=4)
    assert arg.tolist() == [1, 4, 3, 4]          # first occurrence on ties; len(src) for empty segments
    assert val.tolist() == [1.0, 0.0, 5.0, 0.0]


def test_radius_graph_ordering_and_cap():
    torch.manual_seed(0)
    pos = torch.rand(80, 3) * 2.0                  # dense: every node has > 33 candidates
    batch = torch.zeros(80, dtype=torch.long)
    ei = shim.radius_graph(pos, 5.0, batch)
    j, i = ei
    assert torch.all(i[1:] >= i[:-1])
    same = i[1:] == i[:-1]
    assert torch.all(j[1:][same] > j[:-1][same])
    deg = torch.bincount(i, minlength=80)
    # first 33 candidates incl. self: nodes < 33 lose one slot to themselves
    assert deg[:33].eq(32).all() and deg[33:].eq(33).all()
    assert not torch.any(i == j)


@pytest.mark.parametrize("name", ["spherenet_qm9", "dimenetpp_md17", "spherenet_ns3", "schnet_cfg1", "comenet_oc20"])
def test_restated_matches_golden_bitwise(name):
    g, z, pos, batch = case_inputs(name)
    model_name, kw, _, wseed = CASES[name]
    sd = _formula_sd(model_name, kw, wseed)
    if model_name == "SchNet":
        u = restated.schnet_forward(sd, z, pos, batch, cutoff=kw["cutoff"], num_layers=kw["num_layers"])
    elif model_name == "ComENet":
        u = restated.comenet_forward(sd, z, pos, batch, cutoff=kw["cutoff"])
    else:
        u = restated.dimenet_family_forward(sd, z, pos, batch, torsion=(model_name == "SphereNet"),
                                            cutoff=kw["cutoff"], num_spherical=kw.get("num_spherical", 7))
    assert np.array_equal(u.numpy(), g["energy_f32"])


def _formula_sd(model_name, kw, wseed):
    """Key names / shapes come from the fixture's reference run; rebuild them without the reference."""
    import json
    import os
    from helpers import GOLDEN
    with open(os.path.join(GOLDEN, "state_shapes.json")) as fh:
        shapes = json.load(fh)[model_name + json.dumps(kw, sort_keys=True)]
    ref = {k: torch.empty(s) for k, s in shapes.items()}
    if "dist_emb.offset" in ref:
        ref["dist_emb.offset"] = torch.linspace(0.0, kw["cutoff"], shapes["dist_emb.offset"][0])
    return formula_state_dict(ref, seed=wseed)


def test_param_count_known_answer():
    import json
    import os
    from helpers import GOLDEN
    with open(os.path.join(GOLDEN, "state_shapes.json")) as fh:
        shapes = json.load(fh)
    key = "SphereNet" + json.dumps(dict(cutoff=5.0, num_spherical=3), sort_keys=True)
    assert sum(int(np.prod(s)) for s in shapes[key].values()) == 1890118   # threedgraph.ipynb:173


def _live_fixture():
    """Inputs and outputs of the real reference recorded by oracle/gen_golden_live.py."""
    from helpers import GOLDEN
    with open(os.path.join(GOLDEN, "reference_live_shapes.json")) as fh:
        shapes = json.load(fh)
    return load_golden("reference_live"), shapes


@pytest.mark.parametrize("name", ["spherenet_qm9", "dimenetpp_md17"])
def test_restated_matches_live_reference(name):
    """The restatement, with its default basis sizes as the reference model is built for these cases, vs the real
    reference's energies from a run separate from the case fixture's (oracle/gen_golden_live.py); the case fixture
    must hold the same bits."""
    g, z, pos, batch = case_inputs(name)
    live, _ = _live_fixture()
    model_name, kw, _, wseed = CASES[name]
    sd = _formula_sd(model_name, kw, wseed)
    mine = restated.dimenet_family_forward(sd, z, pos, batch, torsion=(model_name == "SphereNet"),
                                           cutoff=kw["cutoff"])
    ref = torch.from_numpy(live["live_" + name])
    assert torch.equal(ref, mine)
    assert torch.equal(ref, torch.from_numpy(g["energy_f32"]))


@pytest.mark.parametrize("name,ctor,wseed", [
    ("pronet_aminoacid", dict(level="aminoacid"), 6),
    ("pronet_backbone", dict(level="backbone", num_blocks=2), 7),
    ("pronet_allatom", dict(level="allatom", num_blocks=2, out_channels=3, out_layers=3), 8)])
def test_pronet_oracle_equals_reference_fixture(name, ctor, wseed):
    """oracle/restated.pronet_forward vs the outputs of the unmodified reference ProNet (fixtures written by
    oracle/gen_golden_pronet.py): energies, edge list and every geometric feature, bit for bit on CPU fp32."""
    import json
    import os
    from helpers import GOLDEN
    from dig_b200.data import Batch
    g = load_golden(name)
    with open(os.path.join(GOLDEN, "state_shapes.json")) as fh:
        shapes = json.load(fh)["ProNet" + json.dumps(ctor, sort_keys=True)]
    sd = formula_state_dict({k: torch.empty(*v) for k, v in shapes.items()}, seed=wseed)
    b = Batch(**{k: torch.from_numpy(g[k]) for k in ("x", "coords_ca", "coords_n", "coords_c", "bb_embs", "side_chain_embs",
                                                    "batch")})
    kw = {k: v for k, v in ctor.items() if k != "out_channels"}
    with torch.no_grad():
        y, inter = restated.pronet_forward(sd, b, return_intermediates=True, **kw)
    assert np.array_equal(inter["edge_index"].numpy(), g["edge_index"])
    for key in ("dist", "theta", "phi", "feature0", "feature1", "pos_emb"):
        assert np.array_equal(inter[key].numpy(), g[key]), key
    assert np.array_equal(y.numpy(), g["energy_f32"])
    assert sum(int(np.prod(v)) for v in shapes.values()) == int(g["num_params"])


NODE_FEATURE_KW = [dict(use_node_features=False), dict(use_extra_node_feature=True, extra_node_feature_dim=3)]


@pytest.mark.parametrize("kw", NODE_FEATURE_KW)
def test_restated_node_feature_options_match_live_reference(kw):
    """spherenet.py:54-91,259-267: the learned shared node embedding and the extra node features, restated vs the real
    reference's energies on the same inputs and weights, bit for bit."""
    g, shapes = _live_fixture()
    i = NODE_FEATURE_KW.index(kw)                  # the order of oracle/gen_golden_live.py
    key = "SphereNet" + json.dumps(dict(cutoff=5.0, num_layers=2, **kw), sort_keys=True)
    sd = formula_state_dict({k: torch.empty(s) for k, s in shapes[key].items()}, seed=11)
    z, pos, batch = (torch.from_numpy(g[f"nodefeat{i}_{k}"]) for k in ("z", "pos", "batch"))
    nf = torch.from_numpy(g[f"nodefeat{i}_node_feature"]) if "extra_node_feature_dim" in kw else None
    with torch.no_grad():
        got = restated.spherenet_forward(sd, z, pos, batch, num_layers=2, node_feature=nf)
    assert torch.equal(got, torch.from_numpy(g[f"nodefeat{i}_energy"]))


def test_restated_gspherenet_geometry_matches_live_reference():
    """oracle.restated.xyztodat_knn vs the outputs of the real ggraph3D/method/G_SphereNet/model/geometric_computing.py
    (run over the shim: the ggraph3D package itself needs rdkit) on the same inputs, bit for bit."""
    g, _ = _live_fixture()
    pos, batch, ei = (torch.from_numpy(g["gsn_" + k]) for k in ("pos", "batch", "edge_index"))
    assert torch.equal(ei, restated.radius_graph(pos, 5.0, batch))    # (the restatement takes target-sorted edge lists)
    got = restated.xyztodat_knn(pos, ei, pos.size(0), batch)
    assert len(got) == int(g["gsn_n_out"])
    for k, out in enumerate(got):
        assert torch.equal(out, torch.from_numpy(g[f"gsn_out{k}"])), k


def _ocp_fixture():
    from dig_b200.data import Batch
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "comenet_ocp.npz"))
    b = Batch(**{k: torch.from_numpy(g[k]) for k in ("atomic_numbers", "pos", "tags", "cell", "edge_index",
                                                     "cell_offsets", "neighbors", "batch")})
    return g, b


def _ocp_formula_sd():
    """Key names / shapes of the OCP model come from the shipped checkpoint's pin (no reference import)."""
    import json
    with open(os.path.join(os.path.dirname(__file__), "golden", "comenet_ocp_checkpoint_shapes.json")) as fh:
        pin = json.load(fh)
    ref = {k[len("module."):]: torch.empty(s) for k, s in pin["keys"].items()}
    sd = formula_state_dict(ref, seed=21)
    sd["lin_out.weight"] = sd["lin_out.weight"] + 0.05
    return sd, pin


def test_restated_comenet_ocp_matches_golden_bitwise():
    """oracle.restated.comenet_ocp_forward vs the fixture written by the UNMODIFIED reference comenet-ocp.py."""
    g, b = _ocp_fixture()
    sd, _ = _ocp_formula_sd()
    u = restated.comenet_ocp_forward(sd, b, cutoff=6.0)
    assert np.array_equal(u.numpy(), g["energy_f32"])


def test_comenet_ocp_state_dict_matches_the_shipped_checkpoint():
    """SURVEY.md 8c golden (4): IS2RETrainedModelWeights.pt has 125 tensors / 4 185 857 parameters; the drop-in class
    built from ocp/comenet.yml exposes exactly those keys and shapes (checkpoint keys carry a `module.` prefix)."""
    from dig_b200.threedgraph.method.comenet_ocp import ComENet
    _, pin = _ocp_formula_sd()
    model = ComENet(0, 0, hidden_channels=256, num_blocks=4, cutoff=6.0, num_radial=3, num_spherical=2, hetero=False,
                    num_output_layers=3)
    mine = {"module." + k: list(v.shape) for k, v in model.state_dict().items()}
    assert mine == pin["keys"] and len(mine) == 125
    assert model.num_params == pin["num_params"] == 4185857
    assert float(model.lin_out.weight.abs().max()) == 0.0          # weight_initializer='zeros'  (comenet-ocp.py:323)
    het = ComENet(0, 0, hidden_channels=256, num_blocks=2, num_radial=3, num_spherical=2, hetero=True)
    assert "interaction_blocks.0.lin.lins.2.weight" in het.state_dict() and het.num_params == 4457731


def test_comenet_ocp_class_loads_the_real_checkpoint():
    """The shipped IS2RE checkpoint, rebuilt from its pinned keys / shapes and a seeded sample of its values (the whole
    embedding table, 16 values of every other tensor, zeros elsewhere), loads strictly and every value lands where the
    checkpoint holds it."""
    from dig_b200.threedgraph.method.comenet_ocp import ComENet
    g, _ = _live_fixture()
    _, pin = _ocp_formula_sd()
    keys = [str(k) for k in g["ckpt_keys"]]
    assert sorted(pin["keys"]) == keys
    state = {k: torch.zeros(s) for k, s in pin["keys"].items()}
    state["module.emb.emb.weight"] = torch.from_numpy(g["ckpt_emb_weight"]).clone()
    for n, i, v in zip(g["ckpt_owner"], g["ckpt_index"], g["ckpt_value"]):
        state[keys[n]].view(-1)[i] = float(v)
    model = ComENet(0, 0, hidden_channels=256, num_blocks=4, cutoff=6.0, num_radial=3, num_spherical=2)
    res = model.load_state_dict(state, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    assert torch.equal(model.emb.emb.weight, torch.from_numpy(g["ckpt_emb_weight"]))
    mine = model.state_dict()
    for n, i, v in zip(g["ckpt_owner"], g["ckpt_index"], g["ckpt_value"]):
        assert float(mine[keys[n][len("module."):]].reshape(-1)[i]) == float(v), keys[n]
