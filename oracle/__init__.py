"""TEST INFRASTRUCTURE ONLY.

`oracle/` holds the checker for the dig.threedgraph hot path:
  * shim.py        pure-torch stand-ins for torch_scatter/torch_sparse/torch_cluster/torch_geometric
  * ref_loader.py  imports the UNMODIFIED reference model code from /root/reference over the shim
                   (only possible where /root/reference exists, i.e. the build container)
  * restated.py    an independent functional restatement of the same algorithms (travels to the GPU box)
  * gen_golden.py  runs the real reference here and writes tests/golden/*.npz

Nothing under dig_b200/ may import this package; only tests/, __graft_entry__.smoke()
and bench.py's cpu_baseline / --impl reference legs do.
"""

# CPU fp32 results of the reference's op sequence depend on how ATen splits its loops and reductions over intra-op
# threads: the fixtures under tests/golden/ are written, and compared bit for bit, with this many threads.  Rewriting
# the case fixtures with 8 threads reproduces every output the tests compare bit for bit (energies, ProNet features),
# while with 1, 2 or 3 threads the energies differ in their last bits.  The reference's CPU forces vary from run to run
# at any thread count (parallel accumulation in its backward); they are compared within a tolerance only.
FIXTURE_THREADS = 8
