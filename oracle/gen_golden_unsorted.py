"""TEST INFRASTRUCTURE ONLY.  Fixture for xyz_to_dat with an edge_index in ARBITRARY order, produced by the unmodified
reference utility (dig/threedgraph/utils/geometric_computing.py:12-80 over oracle/shim.py's SparseTensor):

    python -m oracle.gen_golden_unsorted      ->  tests/golden/xyz_to_dat_unsorted.npz
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle.ref_loader import load_reference_utils  # noqa: E402
from oracle import FIXTURE_THREADS, shim  # noqa: E402
from dig_b200.data import synthetic_batch  # noqa: E402


def main():
    torch.set_num_threads(FIXTURE_THREADS)
    utils = load_reference_utils()
    b = synthetic_batch(3, "qm9", seed=9, variable=True)
    ei = shim.radius_graph(b.pos, 5.0, b.batch)
    gen = torch.Generator().manual_seed(4)
    ei = ei[:, torch.randperm(ei.size(1), generator=gen)].contiguous()
    dist, angle, torsion, i, j, idx_kj, idx_ji = utils.xyz_to_dat(b.pos, ei, b.z.size(0), use_torsion=True)
    out = dict(pos=b.pos.numpy(), edge_index=ei.numpy(), dist=dist.numpy(), angle=angle.numpy(), torsion=torsion.numpy(),
               idx_kj=idx_kj.numpy(), idx_ji=idx_ji.numpy())
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "xyz_to_dat_unsorted.npz"), **out)
    print("E", ei.size(1), "T", idx_kj.numel(), "idx_kj[:6]", idx_kj[:6].tolist(), "idx_ji[:6]", idx_ji[:6].tolist())


if __name__ == "__main__":
    main()
