#!/usr/bin/env python
"""bench.py -- molecules/sec of the SphereNet QM9-shape hot path (BASELINE.json metric, configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--quick] [--dump-outputs DIR]

One "step" = one pass of the hot path (SphereNet 4-layer h=128 forward: radius graph -> geometry ->
basis -> 4 interaction blocks -> readout) over one synthetic batch of 128 QM9-shaped molecules per
GPU (weak scaling: per-GPU work fixed).  Prints ONE JSON line (rank 0).

  value      whole-job molecules/s with the batch already resident in HBM when the timed region starts:
             exactly K steps between barrier + synchronize, CUDA events, max over ranks.  The K-step window is
             repeated (`windows`), `value` is the MEDIAN window and min / max are reported beside it.
  e2e        same metric through the public class API (model(batch)) with HOST (pinned) inputs:
             H2D of z/pos/batch and D2H of the energies inside the timed region, every step
  roofline   the dominant kernel, timed with CUDA events in a separate pass (per entry point of the C ABI) over
             min(K, 10) steps (`roofline.steps`): per-kernel means, not a throughput
  parity     the energies of the timed batches vs the oracle's op sequence on the same GPU (rel err, asserted < 1e-5)
  cpu_baseline  the travelling oracle (oracle/restated.py == the reference's algorithm, bit-identical
             to the real reference on CPU) on this box's host cores, bounded sample
  train      BASELINE configs[4]: forward + backward + overlapped gradient all-reduce + fused Adam step; windows of
             min(max(K, 3), 30) steps (`train.steps`), so that a long headline run does not spend minutes on this
             secondary number
  --impl reference   times that same CPU implementation as the reference arm on the SAME 128-molecule batches, exactly
             K steps after W (at least 1) warm-up steps, ~1.5 s per step
             (the real reference is Python over uninstallable PyG wheels; its restatement is what travels)
  --dump-outputs DIR  after the timed steps, the energies the timed loop returned for its last step (rank 0's
             batch (K - 1) mod 8, float32 [128, 1]) as DIR/energy.npy, in either arm: the inputs and weights are seeded,
             so two builds, or a build and the reference arm, run with the same arguments can be compared output for output
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # no bytecode caches in the tree it runs from, which may be read-only (build() has
                                 # already run there, so the build() call below finds the library up to date)

MOLS_PER_GPU = 128
N_ROTATE = 8                     # distinct batches cycled through the timed region
N_WINDOWS = 5                    # repetitions of the K-step timed window (median reported)
WORKLOAD = "SphereNet 4-layer h=128 (default hparams, ns=7 nr=6), QM9-shape batch=128/GPU (18 atoms, cutoff 5.0), forward"
METRIC = "molecules/sec SphereNet QM9-shape"


def config_block(world):
    """Identical in both arms (the driver compares them)."""
    return {"workload": WORKLOAD, "molecules_per_gpu": MOLS_PER_GPU, "global_batch": MOLS_PER_GPU * world,
            "parallelism": f"graph-sharded x{world} (no data-path collective in inference)",
            "batches": f"{N_ROTATE} distinct synthetic batches rotated (seeds 1000*rank + 0..{N_ROTATE - 1}); "
                       "per-step intermediates (~190 MB) exceed the 126 MB L2",
            "step": "forward (inference) = the headline metric; the training step is under 'train'"}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            p = json.load(fh)
        return p["hbm_gbs"], p.get("bf16_tflops_sustained", p["bf16_tflops"]), "measured"
    return 6650.0, 1400.0, "fallback"


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons DURING the timed region, read in-process through NVML (no fork inside the timed
    window: round 1 forked nvidia-smi every 50 ms on rank 0 and one host hiccup cost a 36 ms window 3x)."""

    def __init__(self, index, period=0.02):
        super().__init__(daemon=True)
        self.index, self.period, self.stop_flag, self.rows = index, period, False, []
        self.nv, self.h = None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
        except Exception:
            self.nv = None

    @staticmethod
    def _physical_index(local):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if local < len(ids) and ids[local].isdigit():
                return int(ids[local])
        return local

    def sample(self):
        nv = self.nv
        if nv is None:
            return
        try:
            sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
            mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
            rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(
                nv, "nvmlDeviceGetCurrentClocksEventReasons") else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            self.rows.append((sm, mx, int(rs)))
        except Exception:
            pass

    def run(self):
        while not self.stop_flag:
            self.sample()
            time.sleep(self.period)

    def summary(self):
        if self.nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": "nvml unavailable"}
        nv = self.nv
        bits = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        sm = [r[0] for r in self.rows]
        reasons = sorted({name for r in self.rows for name, bit in bits.items() if r[2] & bit})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_min_mhz": min(sm) if sm else None,
                "sm_max_mhz": max(r[1] for r in self.rows) if self.rows else None, "reasons": reasons,
                "samples": len(sm), "source": "NVML in-process, sampled during the timed windows"}


def pick_cpu_threads(sd, restated, torch):
    """The reference path is ~9k small ATen ops per forward; with one OpenMP thread per core of a
    128-core host it collapses (measured 0.34 molecules/s).  Try a few thread counts on a tiny
    batch and keep the fastest -- that is "all the host threads it can use"."""
    from dig_b200.data import synthetic_batch
    cores = os.cpu_count() or 1
    tiny = synthetic_batch(4, "qm9", seed=3)
    best, best_t = None, None
    for th in sorted({min(cores, c) for c in (8, 16, 32, cores)}):
        torch.set_num_threads(th)
        with torch.no_grad():
            restated.spherenet_forward(sd, tiny.z, tiny.pos, tiny.batch)
            t0 = time.perf_counter()
            restated.spherenet_forward(sd, tiny.z, tiny.pos, tiny.batch)
            dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = th, dt
        if dt > 20:
            break
    torch.set_num_threads(best)
    return best


def bench_model(torch):
    """The model both arms run: SphereNet defaults, torch.manual_seed(1234) initialisation."""
    from dig_b200.threedgraph.method import SphereNet
    torch.manual_seed(1234)
    return SphereNet()


def bench_batches(rank):
    from dig_b200.data import Batch, synthetic_batch
    out = []
    for sd_ in range(N_ROTATE):        # only what forward() reads travels: z, pos, batch (+ the python int num_graphs)
        full = synthetic_batch(MOLS_PER_GPU, "qm9", seed=1000 * rank + sd_)
        out.append(Batch(z=full.z, pos=full.pos, batch=full.batch, num_graphs=full.num_graphs))
    return out


def cpu_oracle_rate(budget_s=20.0):
    """molecules/s of the CPU restatement of the reference on a bounded sample of the workload (full 128-molecule
    batches of the benchmark, as many forward passes as fit the budget, at least 2)."""
    import torch
    from oracle import restated
    sd = {k: v.detach() for k, v in bench_model(torch).state_dict().items()}
    threads = pick_cpu_threads(sd, restated, torch)
    batches = bench_batches(0)
    with torch.no_grad():
        b = batches[0]
        restated.spherenet_forward(sd, b.z, b.pos, b.batch)          # warm-up
        iters, t0 = 0, time.perf_counter()
        while iters < 2 or (time.perf_counter() - t0 < budget_s and iters < 50):
            b = batches[iters % N_ROTATE]
            restated.spherenet_forward(sd, b.z, b.pos, b.batch)
            iters += 1
        dt = time.perf_counter() - t0
    return MOLS_PER_GPU * iters / dt, dt, iters, threads


def run_reference_arm(args):
    """--impl reference: the reference's own CPU algorithm (oracle port) on the SAME model / batches / batch size,
    all the host threads it can use."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    os.environ["CUDA_VISIBLE_DEVICES"] = ""
    import torch
    from oracle import restated
    sd = {k: v.detach() for k, v in bench_model(torch).state_dict().items()}
    cores = pick_cpu_threads(sd, restated, torch)
    batches = bench_batches(0)
    steps = args.steps
    args.warmup = max(args.warmup, 1)
    with torch.no_grad():
        for s in range(args.warmup):
            b = batches[s % N_ROTATE]
            restated.spherenet_forward(sd, b.z, b.pos, b.batch)
        t0 = time.perf_counter()
        for s in range(steps):
            b = batches[s % N_ROTATE]
            energy = restated.spherenet_forward(sd, b.z, b.pos, b.batch)
        dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, energy)
    val = MOLS_PER_GPU * steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "molecules/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": config_block(world),
            "cpu_baseline": {"value": val, "unit": "molecules/s", "cores": cores, "kind": "port",
                             "host_cores": os.cpu_count(),
                             "sample": f"{steps} forward passes over the benchmark's {MOLS_PER_GPU}-molecule QM9-shape "
                                       "batches (oracle/restated.py, bit-identical to the reference on CPU)"},
            "e2e": {"value": val, "unit": "molecules/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def dump_outputs(out_dir, energy):
    """--dump-outputs: the energies of the last timed step as out_dir/energy.npy, float32."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "energy.npy"), energy.detach().cpu().numpy().astype(np.float32))


def time_ms(torch, fn, n=10, warm=3):
    for _ in range(warm):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def other_configs(dev):
    """BASELINE.json configs[0], [2], [3] (parity-test cases, not the headline): short CUDA-event timings of the
    inference forward, the energy+force forward where the config asks for forces, and one training step, so that every
    configured mode has a measured number (SURVEY.md 8d).  Errors are reported in the JSON, not swallowed."""
    import torch
    from dig_b200.data import synthetic_batch, synthetic_proteins
    from dig_b200.threedgraph.method import ComENet, DimeNetPP, ProNet, SchNet

    cases = [("cfg1 SchNet 2-layer h=32, 16 x 12 atoms, cutoff 10",
              lambda f: SchNet(energy_and_force=f, num_layers=2, hidden_channels=32, num_filters=32, cutoff=10.0),
              dict(nmol=16, shape="schnet-plumbing", seed=0), True),
             ("cfg3 DimeNet++ 4-block h=128, MD17-aspirin-shape batch=256, energy+force",
              lambda f: DimeNetPP(energy_and_force=f, cutoff=5.0), dict(nmol=256, shape="md17-aspirin", seed=3), True),
             ("cfg4 ComENet 4-layer h=256, OC20-IS2RE-shape batch=64, cutoff 6.0",
              lambda f: ComENet(cutoff=6.0), dict(nmol=64, shape="oc20-is2re", seed=4), False),
             ("next row (SURVEY 8f-1): ProNet aminoacid level, 32 synthetic proteins x ~100 residues, cutoff 10",
              lambda f: ProNet(level="aminoacid"), dict(protein=True, nmol=32), False)]
    out = []
    for name, make, data_kw, forces in cases:
        rec = {"config": name}
        try:
            torch.manual_seed(7)
            if data_kw.get("protein"):
                b = synthetic_proteins(data_kw["nmol"], length=100, seed=5).to(dev)
            else:
                b = synthetic_batch(**data_kw).to(dev)
            nmol = data_kw["nmol"]
            model = make(False).to(dev)

            def infer():
                with torch.no_grad():
                    return model(b)
            ms = time_ms(torch, infer)
            rec["inference"] = {"ms_per_step": round(ms, 4), "molecules_per_s": round(nmol / (ms * 1e-3), 1)}
            if not data_kw.get("protein"):
                # the same forward with batches in flight (dig_b200.pipeline, what run.val does)
                from dig_b200.pipeline import InferencePipeline
                pipe = InferencePipeline(model.eval(), dev)
                for _ in pipe.map([b] * (2 * pipe.depth)):
                    pass
                ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                ea.record()
                n_rep = 12
                for _ in pipe.map([b] * n_rep):
                    pass
                cur = torch.cuda.current_stream()
                for st in pipe.streams:
                    cur.wait_stream(st)
                eb.record()
                torch.cuda.synchronize()
                msp = ea.elapsed_time(eb) / n_rep
                rec["inference"]["in_flight"] = {"batches": pipe.depth, "ms_per_step": round(msp, 4),
                                                 "molecules_per_s": round(nmol / (msp * 1e-3), 1)}
                model.train()
            # whole-forward roofline view (SURVEY 8d flop counts; fp32 work counted once): which pipe would bound it
            from dig_b200 import ops as _ops
            if hasattr(b, "pos") and not data_kw.get("protein"):
                gg = _ops.build_graph(b.pos, b.batch, model.cutoff, num_graphs=nmol)
                E_, N_ = gg.n_edges, gg.n_nodes
                fl = None
                if name.startswith("cfg4"):          # ComENet: 1.70 MFLOP/node + 68.8 kFLOP/edge per block, 4 blocks
                    fl = 4 * (N_ * 1.70e6 + E_ * 68.8e3)
                    kind = "tcgen05 3xFP16 engine for the hidden x hidden linears (dig3d_linear_h16) + FP32 edge-filter aggregation"
                elif name.startswith("cfg3"):        # DimeNet++: 331 kFLOP/edge + 2.8 kFLOP/triplet per block + node MLPs
                    _ops.triplet_geometry(gg, b.pos, use_torsion=False, want_idx=False)
                    fl = 4 * (E_ * 331e3 + gg.n_triplets * 2.8e3) + 5 * N_ * 459e3
                    kind = "tcgen05 3xFP16 dense chain + FP32 triplet kernels"
                elif name.startswith("cfg1"):        # SchNet: 2(G F + F^2) + 3F per edge, 2(HF + FH + H^2) per node, 2 layers
                    fl = 2 * (E_ * (2 * (50 * 32 + 32 * 32) + 96) + N_ * 2 * 3 * 32 * 32)
                    kind = "fp32 FFMA (launch-latency bound at this size)"
                if fl:
                    rec["inference"]["roofline"] = {"flops_per_step": fl, "achieved_tflops": round(fl / (ms * 1e-3) / 1e12, 3),
                                                    "frac_of_tensor_peak": round(fl / (ms * 1e-3) / 1e12 / peaks()[1], 5),
                                                    "edges": E_, "nodes": N_, "pipe": kind}
            y = torch.randn(nmol, 1, device=dev)
            opt = torch.optim.Adam(model.parameters(), lr=5e-4)

            def train():
                opt.zero_grad()
                torch.nn.functional.l1_loss(model(b), y).backward()
                opt.step()
            ms = time_ms(torch, train, n=5)
            rec["train_step"] = {"ms_per_step": round(ms, 4), "molecules_per_s": round(nmol / (ms * 1e-3), 1)}
            if forces:
                fmodel = make(True).to(dev)
                fmodel.load_state_dict(model.state_dict())
                fmodel.eval()

                def ef():
                    b.pos.grad = None
                    o = fmodel(b)
                    return torch.autograd.grad(o, b.pos, grad_outputs=torch.ones_like(o))[0]
                ms = time_ms(torch, ef, n=5)
                rec["energy_and_force"] = {"ms_per_step": round(ms, 4), "molecules_per_s": round(nmol / (ms * 1e-3), 1)}
                # training ON forces (reference run.py:110-123): loss = L1(E) + 100 L1(F), F = -dE/dpos under create_graph
                fmodel.train()
                fopt = torch.optim.Adam(fmodel.parameters(), lr=5e-4)
                f_t = torch.randn(b.pos.size(0), 3, device=dev)

                def ftrain():
                    fopt.zero_grad()
                    b.pos.grad = None
                    o = fmodel(b)
                    force = -torch.autograd.grad(o, b.pos, grad_outputs=torch.ones_like(o), create_graph=True,
                                                 retain_graph=True)[0]
                    loss = torch.nn.functional.l1_loss(o, y) + 100.0 * torch.nn.functional.l1_loss(force, f_t)
                    loss.backward()
                    fopt.step()
                ms = time_ms(torch, ftrain, n=3)
                rec["force_train_step"] = {"ms_per_step": round(ms, 4), "molecules_per_s": round(nmol / (ms * 1e-3), 1),
                                           "what": "energy + force loss, second-order path (tangent network)"}
                b.pos.requires_grad_(False)
        except Exception as exc:                      # reported, never hidden
            rec["error"] = f"{type(exc).__name__}: {exc}"
        out.append(rec)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="headline + roofline only (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the energies of the last timed step as DIR/energy.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference_arm(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # keep stdout to the one JSON line: some environments export NCCL_DEBUG=VERSION, which makes NCCL print its
        # version banner on stdout at communicator creation
        os.environ.setdefault("NCCL_DEBUG", "WARN")
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)
    import __graft_entry__
    if rank == 0:
        __graft_entry__.build()
    if world > 1:
        dist.barrier()
    from dig_b200 import _lib, ops
    from dig_b200.threedgraph.method import SphereNet

    model = bench_model(torch).to(dev).eval()
    host = [b.pin_memory() for b in bench_batches(rank)]
    resident = [b.to(dev) for b in host]
    h2d = sum(getattr(host[0], k).numel() * getattr(host[0], k).element_size() for k in ("z", "pos", "batch"))
    d2h = MOLS_PER_GPU * 4

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps, join=None):
        """Exactly `steps` steps between barrier + synchronize on both sides; (device ms, wall ms), max over ranks.
        `join` makes the timing stream wait for the side streams of a pipelined loop before the closing event."""
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        a.record()
        for s in range(steps):
            fn(s)
        if join is not None:
            join()
        b.record()
        barrier()
        wall = time.perf_counter() - t0
        ms = torch.tensor([a.elapsed_time(b), wall * 1e3], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms[0]), float(ms[1])

    def windows(fn, steps, n=N_WINDOWS, join=None):
        res = [timed(fn, steps, join) for _ in range(n)]
        dev_ms = sorted(r[0] for r in res)
        wall_ms = sorted(r[1] for r in res)
        return dev_ms, wall_ms

    sink = []

    def step_resident(s):
        with torch.no_grad():
            sink.append(model(resident[s % N_ROTATE]))
        if len(sink) > 4:
            sink.pop(0)

    out_host = torch.empty(MOLS_PER_GPU, 1, dtype=torch.float32).pin_memory()

    def step_e2e(s):
        hb = host[s % N_ROTATE]
        with torch.no_grad():
            db = hb.to(dev, non_blocking=True)
            u = model(db)
            out_host.copy_(u, non_blocking=True)
        torch.cuda.current_stream().synchronize()      # the user reads the energies every step

    # the same loop with `depth` batches in flight (dig_b200.pipeline.InferencePipeline, what run.val does): every step still
    # copies its inputs from pinned host memory and its energies are still read on the host, one step later
    from dig_b200.pipeline import InferencePipeline
    from dig_b200.pipeline import DEFAULT_DEPTH
    depth = max(1, int(os.environ.get("DIG3D_BENCH_STREAMS", str(DEFAULT_DEPTH))))
    pipe = InferencePipeline(model, dev, depth=depth)
    pipe_r = InferencePipeline(model, dev, depth=depth)
    pending, pending_r = [], []
    checksum = [0.0]
    last_r = [None]                                       # host energies of the latest step step_resident_pipelined took

    def step_e2e_pipelined(s):
        pending.append(pipe.submit(host[s % N_ROTATE]))
        last = (s == args.steps - 1)
        while len(pending) > (0 if last else depth - 1):
            checksum[0] += float(pipe.result(pending.pop(0))[0, 0])     # the host reads an earlier step's energies

    def step_resident_pipelined(s):
        """The device-resident loop with `depth` batches in flight (the tail of one batch's kernels overlaps the head of
        the next on another stream); the K steps of a window are all complete before its closing event."""
        pending_r.append(pipe_r.submit(resident[s % N_ROTATE]))
        last = (s == args.steps - 1)
        while len(pending_r) > (0 if last else depth - 1):
            last_r[0] = pipe_r.result(pending_r.pop(0))

    def join_streams():
        cur = torch.cuda.current_stream()
        for p_ in (pipe, pipe_r):
            for st in p_.streams:
                cur.wait_stream(st)

    for s in range(args.warmup):
        step_resident(s)
        step_e2e(s)
    for s in list(range(max(args.warmup, 3) + 2 * depth)) + [args.steps - 1]:
        step_e2e_pipelined(s)                            # warm the side streams' allocator pools; the last call flushes
    for s in list(range(max(args.warmup, 3) + 2 * depth)) + [args.steps - 1]:
        step_resident_pipelined(s)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = _lib.launch_count
    dev_w, wall_w = windows(step_resident, args.steps)
    launches = (_lib.launch_count - l0) // N_WINDOWS
    e2e_dev_w, e2e_wall_w = windows(step_e2e, args.steps)
    _, e2e_pipe_wall_w = windows(step_e2e_pipelined, args.steps, join=join_streams)
    dev_serial_w = dev_w
    if depth > 1:
        dev_w, wall_w = windows(step_resident_pipelined, args.steps, join=join_streams)
    sampler.stop_flag = True
    if args.dump_outputs and rank == 0:
        # what the loop behind `value` returned for its last timed step (pipe_r takes no further batches, so its host
        # buffer still holds them)
        dump_outputs(args.dump_outputs, last_r[0] if depth > 1 else sink[-1])
    ms = statistics.median(dev_w)
    ms_serial = statistics.median(dev_serial_w)
    wall_e2e_serial = statistics.median(e2e_wall_w)
    wall_e2e = statistics.median(e2e_pipe_wall_w)
    total_mols = MOLS_PER_GPU * world * args.steps
    value = total_mols / (ms * 1e-3)
    e2e = total_mols / (wall_e2e * 1e-3)          # wall clock: includes host work and the per-step sync
    overflow = ops.h16_overflow(clear=True)

    # ---- training step (BASELINE configs[4]): forward + backward kernels, overlapped NCCL gradient all-reduce over the
    #      flat gradient buffer, fused Adam.  Secondary number (the headline metric is inference throughput).
    train = None
    if not args.quick:
        from dig_b200 import parallel
        torch.manual_seed(4321)
        tmodel = SphereNet().to(dev)
        flat = parallel.FlatParameters(tmodel)
        topt = parallel.FlatAdam(flat, lr=5e-4)
        reducer = parallel.GradientReducer(flat)
        gen = torch.Generator().manual_seed(99 + rank)
        targets = [torch.randn(MOLS_PER_GPU, 1, generator=gen).to(dev) for _ in range(N_ROTATE)]
        l1 = torch.nn.L1Loss()

        def step_train(s):
            flat.zero_grad()
            reducer.arm()
            out = tmodel(resident[s % N_ROTATE])
            loss = l1(out, targets[s % N_ROTATE])
            loss.backward()
            reducer.finish()
            topt.step()

        train_steps = max(3, min(args.steps, 30))
        with parallel.PacedGC(every=0):                  # as run.train does: no rank pauses for cycle collection mid-window
            for s in range(3):
                step_train(s)
            lt0 = _lib.launch_count
            tr_dev, _ = windows(step_train, train_steps, n=3)
        train_launches = (_lib.launch_count - lt0) // 3
        ms_train = statistics.median(tr_dev)
        train = {"value": MOLS_PER_GPU * world * train_steps / (ms_train * 1e-3), "unit": "molecules/s",
                 "ms_per_step": ms_train / train_steps, "steps": train_steps, "gpu_launches": train_launches,
                 "windows_ms_per_step": [round(w / train_steps, 4) for w in tr_dev],
                 "allreduce_bytes_per_step": reducer.bytes_per_step if world > 1 else 0,
                 "step": "SphereNet forward + backward (dig_b200/autograd.py kernels) + gradient all-reduce "
                         "(flat buffer, launched from autograd hooks on a side stream under the backward tail) + "
                         "fused Adam kernel, L1 loss on synthetic targets"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline pass: per-kernel CUDA events (separate pass so the events do not perturb `value`)
    hbm_peak, tf_peak, which = peaks()
    n_roof = min(args.steps, 10)
    _lib.start_timing()
    for s in range(n_roof):
        step_resident(s)
    per = _lib.stop_timing()
    gr = ops.build_graph(resident[0].pos, resident[0].batch, 5.0, num_graphs=MOLS_PER_GPU)
    E, T, N = gr.n_edges, gr.n_triplets, gr.n_nodes
    H, I = 128, 64
    kern = {k: sum(v) / len(v) for k, v in per.items()}
    total_by_kernel = {k: sum(v) / n_roof for k, v in per.items()}
    step_kernel_ms = sum(total_by_kernel.values())
    dom = max(total_by_kernel, key=total_by_kernel.get)
    dom_ms = kern[dom]
    # algorithmic work per launch of the kernels that can dominate (DESIGN.md "kernels")
    work = {
        # chain B: lin_up + 7 (128x128) linears; reads m, x_ji, e1_in, rbf0, dst; writes e1_out, v_in
        "dig3d_sphere_update_e_b_h16": (E * (2 * I * H + 7 * 2 * H * H), 4 * (E * (I + 3 * H + 6 + 1) + N * H), "tensor"),
        "dig3d_sphere_update_e_b_tc": (E * (2 * I * H + 7 * 2 * H * H), 4 * (E * (I + 3 * H + 6 + 1) + N * H), "tensor"),
        # chain B of block l + part A of block l + 1 in one launch (e1 stays on chip between them)
        "dig3d_sphere_update_e_ba_h16": (E * (2 * I * H + 7 * 2 * H * H) + E * (2 * 2 * H * H + 2 * H * I),
                                         4 * (E * (I + 3 * H + 6 + 1) + N * H) + 4 * E * (H + I), "tensor"),
        "dig3d_sphere_update_e_a_h16": (E * (2 * 2 * H * H + 2 * H * I), 4 * E * (H + H + I + 6), "tensor"),
        "dig3d_sphere_update_e_a_tc": (E * (2 * 2 * H * H + 2 * H * I), 4 * E * (H + H + I + 6), "tensor"),
        "dig3d_sphere_init_e_h16": (E * 2 * 3 * H * H, 4 * (E * (H + 6 + 2) + N * H), "tensor"),
        # triplet gather: x_down rows once per edge (staged), 16 projected-basis floats per triplet, m out
        "dig3d_sphere_triplet_gather_node": (T * (2 * 2 * 8 * I + 3 * I), 4 * (E * I + T * 16 + E * I), "hbm"),
        "dig3d_sphere_triplet_gather": (T * (2 * 2 * 8 * I + 3 * I), 4 * (E * I + T * 16 + E * I), "hbm"),
        "dig3d_sphere_triplet_gather_warp": (T * (2 * 2 * 8 * I + 3 * I), 4 * (E * I + T * 16 + E * I), "hbm"),
        "dig3d_triplet_basis_project": (2 * (E * 336 * 32 + T * 56 * 32), 4 * (E * 42 + 2 * T + 64 * T), "hbm"),
        "dig3d_triplet_basis_project_lists": (2 * (E * 336 * 32 + T * 56 * 32), 4 * (E * 42 + 2 * T + 64 * T), "hbm"),
        "dig3d_sphere_update_v_batched": (5 * 2 * N * (128 * 256 + 3 * 256 * 256 + 256), 4 * 5 * N * (H + 1), "tensor"),
        "dig3d_sphere_update_v_h16": (5 * 2 * N * (128 * 256 + 3 * 256 * 256 + 256), 4 * 5 * N * (H + 1), "tensor"),
    }
    flops_d, bytes_d, bound = work.get(dom, (0, 0, "hbm"))
    calls_per_step = len(per[dom]) / n_roof
    traffic_file = os.path.join(ROOT, "profiles", "r02_dram_traffic.json")
    traffic = None
    if os.path.exists(traffic_file):
        with open(traffic_file) as fh:
            traffic = json.load(fh).get(dom.replace("dig3d_", ""))
    ach = (flops_d / (dom_ms * 1e-3) / 1e12) if bound == "tensor" else (bytes_d / (dom_ms * 1e-3) / 1e9)
    peak = tf_peak if bound == "tensor" else hbm_peak
    roof = {"kernel": dom.replace("dig3d_", ""), "steps": n_roof, "bound": bound, "achieved": ach, "peak": peak,
            "unit": "TFLOP/s" if bound == "tensor" else "GB/s", "frac": ach / peak if peak else None,
            "traffic": traffic, "traffic_source": "profiles/r02_dram_traffic.json (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per launch)" if traffic else None,
            "peak_source": f"{which} " + ("bf16_tflops_sustained (kernel timed inside the step; kind::f16 MMAs run at the bf16 rate)" if bound == "tensor" else "hbm_gbs"),
            "ms_per_launch": dom_ms, "launches_per_step": calls_per_step,
            "share_of_step_kernel_time": total_by_kernel[dom] / step_kernel_ms,
            "algorithmic_flops_per_launch": flops_d, "algorithmic_bytes_per_launch": bytes_d,
            "note": "flops counted once per fp32 product; the tensor-core chains issue 3 MMAs per product (hi/lo split "
                    "operands for 1e-5 parity), so the tensor pipe does 3x this work -- see tensor_pipe_frac",
            "tensor_pipe_frac": (3 * ach / peak) if bound == "tensor" else None,
            "kernel_ms": {k.replace("dig3d_", ""): round(v, 5) for k, v in sorted(kern.items())},
            "per_step_ms": {k.replace("dig3d_", ""): round(v, 5) for k, v in sorted(total_by_kernel.items())}}
    # the tensor chain of update_e part B is reported in every run (it was the round-1 dominant kernel)
    for name in ("dig3d_sphere_update_e_b_h16", "dig3d_sphere_update_e_b_tc"):
        if name in kern:
            fl, by, _ = work[name]
            t_ach = fl / (kern[name] * 1e-3) / 1e12
            roof["update_e_b"] = {"kernel": name.replace("dig3d_", ""), "ms_per_launch": kern[name], "achieved": t_ach,
                                  "peak": tf_peak, "unit": "TFLOP/s", "frac": t_ach / tf_peak,
                                  "tensor_pipe_frac": 3 * t_ach / tf_peak,
                                  "hbm_view": {"achieved": by / (kern[name] * 1e-3) / 1e9, "peak": hbm_peak,
                                               "unit": "GB/s", "frac": by / (kern[name] * 1e-3) / 1e9 / hbm_peak}}
            break

    # ---- scatter (segment-sum) HBM roofline: the second half of BASELINE.json's metric
    rep = 48
    ptr = torch.cat([gr.row_ptr[:-1].to(torch.int64) + r * E for r in range(rep)] +
                    [torch.tensor([rep * E], device=dev)]).to(torch.int32)
    x = torch.randn(rep * E, H, device=dev)
    seg_ms = time_ms(torch, lambda: ops.segment_sum(x, ptr), n=10, warm=3)
    seg_bytes = 4 * (rep * E * H + rep * N + rep * N * H)
    scatter = {"kernel": "segment_sum_kernel", "rows": rep * E, "width": H, "segments": rep * N,
               "bytes": seg_bytes, "ms": seg_ms, "achieved": seg_bytes / (seg_ms * 1e-3) / 1e9,
               "peak": hbm_peak, "unit": "GB/s", "frac": seg_bytes / (seg_ms * 1e-3) / 1e9 / hbm_peak,
               "input_mb": rep * E * H * 4 / 1e6}
    del x

    # ---- parity on the timed batches + GPU comparator (BASELINE.md section 3): the reference's op sequence
    #      (oracle/restated.py == the reference code over torch-native scatter) executed by ATen/cuBLAS on this B200
    gpu_cmp, parity = None, None
    if world == 1 and not args.quick:
        from oracle import restated
        sd_dev = {k: v.detach() for k, v in model.state_dict().items()}
        worst = 0.0
        with torch.no_grad():
            for rb in resident:
                ref = restated.spherenet_forward(sd_dev, rb.z, rb.pos, rb.batch, num_graphs=MOLS_PER_GPU)
                got = model(rb)
                worst = max(worst, float((got - ref).abs().max() / ref.abs().max()))
        parity = {"rel_err_max": worst, "tolerance": 1e-5, "batches": N_ROTATE,
                  "what": "max |E - E_oracle| / max |E_oracle| over the timed batches, oracle op sequence on the same GPU",
                  "fp16_range_overflow": bool(overflow)}
        assert worst < 1e-5 and not overflow, f"parity on the timed batches failed: {parity}"
        it = [0]

        def ref_step():
            rb_ = resident[it[0] % N_ROTATE]
            it[0] += 1
            with torch.no_grad():
                restated.spherenet_forward(sd_dev, rb_.z, rb_.pos, rb_.batch, num_graphs=MOLS_PER_GPU)
        ms_ref = time_ms(torch, ref_step, n=10, warm=2)
        gpu_cmp = {"value": MOLS_PER_GPU / (ms_ref * 1e-3), "unit": "molecules/s", "ms_per_step": ms_ref,
                   "timing": "CUDA events, 10 iterations after 2 warm-ups",
                   "what": "reference op sequence (oracle/restated.py) on the same B200 through ATen/cuBLAS fp32, "
                           "torch-native scatter; same batches and weights"}

        # the same for a training step: torch.autograd over the reference op sequence + Adam
        sd_t = {k: v.detach().clone().requires_grad_(v.is_floating_point()) for k, v in tmodel.state_dict().items()}
        ropt = torch.optim.Adam([v for v in sd_t.values() if v.requires_grad], lr=5e-4)
        jt = [0]

        def ref_train():
            s_ = jt[0]
            jt[0] += 1
            rb_ = resident[s_ % N_ROTATE]
            ropt.zero_grad()
            o = restated.spherenet_forward(sd_t, rb_.z, rb_.pos, rb_.batch, num_graphs=MOLS_PER_GPU)
            l1(o, targets[s_ % N_ROTATE]).backward()
            ropt.step()
        ms_rt = time_ms(torch, ref_train, n=5, warm=1)
        train["gpu_comparator"] = {"value": MOLS_PER_GPU / (ms_rt * 1e-3), "unit": "molecules/s", "ms_per_step": ms_rt,
                                   "what": "torch.autograd over the reference op sequence + Adam on the same B200"}
        del sd_t, ropt

    others = other_configs(dev) if (world == 1 and not args.quick) else None

    cpu = None
    if world == 1 and not args.no_cpu_baseline and not args.quick:
        rate, dt, iters, threads = cpu_oracle_rate()
        cpu = {"value": rate, "unit": "molecules/s", "cores": threads, "kind": "port",
               "host_cores": os.cpu_count(),
               "sample": f"{iters} forward passes over the benchmark's {MOLS_PER_GPU}-molecule QM9-shape batches ({dt:.1f} s), "
                         "oracle/restated.py (bit-identical to the reference's CPU path); thread count = fastest of {8,16,32,all}"}

    per_step = [w / args.steps for w in dev_w]
    line = {"metric": METRIC, "value": value, "unit": "molecules/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": config_block(world),
            "windows": {"n": N_WINDOWS, "steps_each": args.steps, "ms_per_step_min": per_step[0],
                        "ms_per_step_median": statistics.median(per_step), "ms_per_step_max": per_step[-1],
                        "rule": "value = the median window; each window = exactly K steps (batches_in_flight of them overlapping on alternating streams) between barrier + synchronize, all K complete before the closing event, max over ranks"},
            "sizes": {"edges": E, "triplets": T, "nodes": N},
            "batches_in_flight": depth,
            "serial": {"value": total_mols / (ms_serial * 1e-3), "ms_per_step": ms_serial / args.steps,
                       "what": "one batch at a time on one stream (the loop the per-kernel roofline entries are timed in)"},
            "e2e": {"value": e2e, "unit": "molecules/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": wall_e2e / args.steps, "ms_per_step_min": e2e_pipe_wall_w[0] / args.steps,
                    "ms_per_step_max": e2e_pipe_wall_w[-1] / args.steps,
                    "api": f"dig_b200.pipeline.InferencePipeline (the loop of run.val): {depth} batches in flight on "
                           "alternating streams; every step copies its inputs from pinned host memory and its energies are "
                           "read on the host a step or two later",
                    "serial": {"value": total_mols / (wall_e2e_serial * 1e-3), "ms_per_step": wall_e2e_serial / args.steps,
                               "api": "model(batch.to(device)) + .copy_ to a pinned buffer + stream sync every step"},
                    "timing": "host wall clock over exactly K steps (barrier + synchronize on both sides), median of the windows"},
            "gpu_launches": launches, "wall_ms_per_step": statistics.median(wall_w) / args.steps,
            "clocks": sampler.summary(), "roofline": roof, "scatter_roofline": scatter, "parity": parity,
            "cpu_baseline": cpu, "gpu_comparator": gpu_cmp, "other_configs": others, "train": train}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
