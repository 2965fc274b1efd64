#!/usr/bin/env python
"""Benchmark of the ANI-2x energy+force hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--config NAME] [--dump-outputs DIR]     # B200 arm (this repo)
    python bench.py --impl reference --steps K --warmup W [--config NAME]
                                      # reference arm: the UNMODIFIED aiqm/torchani on the host cores

One "step" = energy AND forces of the whole system (neighbour search -> AEV -> 8-member MLP ensemble ->
forces).  Configurations (BASELINE.json `configs`, SURVEY.md 8d), seeded synthetic coordinates and weights:

    water10k    (default; the configuration the metric is quoted on)  ANI-2x x8, periodic 9999-atom water box
    water1k     periodic 999-atom water box
    gdb256      batch of 256 GDB-11-like conformers (9-26 atoms, H/C/N/O, -1 padding, no PBC, all-pairs semantics)
    protein50k  1C17 protein (H C N O S) + lattice water, 50k atoms, periodic, through the host calculator

Metric: atom-steps/s (= real atoms / t_step; ns/day at 1 fs = 0.0864 / t_step and conformers/s are reported too).
With N > 1 GPUs (torchrun, one rank per GPU) the SAME system is sharded over the ranks by central atom (strong
scaling); the partial forces / energies are summed on the device over NVLink peer memory by one kernel inside the
step's CUDA graph (torchani_b200/csrc/comm.cu).

Timing: W >= 3 warm-up steps, then K steps each bracketed by CUDA events on the launch stream; between timed steps
a 256 MiB buffer is overwritten (L2 flush, untimed); barrier + synchronize on both sides of the region; per-step
times are summed, max over ranks.  `e2e` = the same metric through the host-buffer API (pinned host positions in,
host energy + forces out, copies inside the timed region).  Prints ONE JSON line on rank 0.

Reference arm (`--impl reference`): the real reference package (oracle/_ref/torchani, staged by
oracle/build_ref.sh) on the CPU -- strategy="pyaev", neighborlist="cell_list" (single periodic system) or
"all_pairs" (batch), python Ensemble loop, float32, torchani.grad.energies_and_forces -- with one thread per
PHYSICAL core; every step is one full evaluation of the same workload; the run stops early (>= 1 timed step)
when its time budget is spent.  Where the staged reference is missing the CPU port of its algorithm
(oracle/ani_oracle.py) is timed instead and the line says `kind: "port"`.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "ani2x_energy_force_atom_steps_per_s"
UNIT = "atom-steps/s"
# SURVEY.md 8(d): algorithmic bytes per atom of the AEV kernels (fp32, ANI-2x)
AEV_FWD_BYTES_PER_ATOM = 4276.0
AEV_BWD_BYTES_PER_ATOM = 4288.0

CONFIGS = {
    "water10k": "ANI-2x x8 ensemble, periodic water box, 9999 atoms (BASELINE configs[3]), energy+forces per step",
    "water1k": "ANI-2x x8 ensemble, periodic water box, 999 atoms (BASELINE configs[1]), energy+forces per step",
    "gdb256": "ANI-2x x8 ensemble, batch of 256 GDB-11-like conformers, 9-26 atoms each, H/C/N/O, -1 padding, no "
              "PBC (BASELINE configs[2], training-benchmark shapes), energies+forces of the batch per step",
    "protein50k": "ANI-2x x8 ensemble, 1C17 protein (H C N O S, cut to the box) in lattice water, ~50k atoms, cubic "
                  "periodic box 79.4 A (BASELINE configs[4]), energy+forces per step through the host calculator",
}


def make_workload(name: str, molecules: int = 0):
    """-> dict(z, idx, coords, cell, pbc, n_atoms (real), n_conf, batch)"""
    from torchani_b200 import synthetic
    if name in ("water10k", "water1k"):
        n_mol = molecules or (3333 if name == "water10k" else 333)
        z, idx, coords, cell, pbc = synthetic.water_box(n_mol, seed=0)
    elif name == "protein50k":
        z, idx, coords, cell, pbc = synthetic.protein_in_water(50001, seed=0)
    elif name == "gdb256":
        idx, coords = synthetic.conformer_batch(256, seed=1234)
        conv = torch.tensor([1, 6, 7, 8])
        z = torch.where(idx >= 0, conv[idx.clamp(min=0)], torch.full_like(idx, -1))
        cell = pbc = None
    else:
        raise ValueError(name)
    return {"z": z, "idx": idx, "coords": coords, "cell": cell, "pbc": pbc, "n_atoms": int((idx >= 0).sum()),
            "n_conf": int(idx.shape[0]), "batch": name == "gdb256"}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"], "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "source": "fallback (B200_PROFILING.md)"}


def library_hash() -> str:
    from torchani_b200 import _lib
    h = hashlib.sha256()
    with open(_lib.LIB_PATH, "rb") as fh:
        h.update(fh.read())
    return h.hexdigest()[:16]


def library_build_id() -> str:
    """Fingerprint of the sources + flags the library on disk was built from (torchani_b200.build.build_id)."""
    from torchani_b200 import build as _build
    return _build.build_id()


def measured_traffic(config: str):
    """dram bytes per launch from an `ncu --set full` capture OF THE LIBRARY BUILD BEING RUN: profiles/traffic.json maps
    kernel build id (fingerprint of the sources + flags the AEV / GEMM kernels are compiled from; nvcc output is not
    byte-reproducible), build id or library hash -> config -> {mlp, aev_forward, aev_backward}; anything else is null
    (never a stale literal)."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(path):
        return {}
    try:
        data = json.load(open(path))
        from torchani_b200 import build as _build
        for key in (_build.build_id(kernels_only=True), library_build_id(), library_hash()):
            if key and key in data:
                return data[key].get(config, {})
        return {}
    except (OSError, ValueError):
        return {}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms during the timed region."""

    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
            t0 = time.time()
            while not self.rows and time.time() - t0 < 5.0:   # nvidia-smi takes a moment to start sampling
                time.sleep(0.05)
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([v.strip() for v in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) > 2 + k and r[2 + k] == "Active" for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------
# the reference on the host cores
# ---------------------------------------------------------------------------------------------------------
def physical_cores() -> int:
    try:
        import psutil
        n = psutil.cpu_count(logical=False)
        if n:
            return int(n)
    except Exception:
        pass
    return max(1, (os.cpu_count() or 2) // 2)


def run_cpu_reference(work, steps: int, warmup: int, budget_s: float):
    """Times the reference's own CPU implementation on this workload.  -> (per-step seconds, kind, threads, what)."""
    threads = physical_cores()
    torch.set_num_threads(threads)   # torchrun pins OMP_NUM_THREADS=1: undo that for the CPU arm
    z, coords, cell, pbc = work["z"], work["coords"], work["cell"], work["pbc"]
    try:
        import oracle.ref_torchani as rt
        if not rt.available():
            raise ImportError("oracle/_ref/torchani is not staged")
        from torchani_b200 import models, synthetic
        weights = synthetic.make_weights(models.SYMBOLS_2X, synthetic.DIMS_2X, 1008, 8, seed=1234)
        nl = "all_pairs" if work["batch"] else "cell_list"
        model = rt.build_model(weights, "2x", "cpu", strategy="pyaev", neighborlist=nl)
        kind = "reference"
        what = (f"unmodified aiqm/torchani (oracle/_ref/torchani): strategy=pyaev, neighborlist={nl}, python Ensemble "
                f"loop, float32, torchani.grad.energies_and_forces")

        def step():
            return rt.energies_and_forces(model, z, coords.clone(), cell, pbc)
    except Exception as exc:   # the staged package is absent on this box: the CPU port of the same algorithm
        import oracle.ani_oracle as orc
        model = orc.ani2x_model(seed=1234, members=8, neighborlist="all_pairs" if work["batch"] else "cell_list")
        kind = "port"
        what = f"CPU port of the reference algorithm (oracle/ani_oracle.py, float32) [{type(exc).__name__}: {exc}]"
        idx = work["idx"]

        def step():
            out = orc.compute(model, idx, coords, cell, pbc, forces=True)
            return out["energy"], out["forces"]

    t_begin = time.perf_counter()
    for _ in range(warmup):
        step()
        if time.perf_counter() - t_begin > budget_s / 3:
            break
    times = []
    for _ in range(max(1, steps)):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_begin > budget_s:
            break
    return times, kind, torch.get_num_threads(), what


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="water10k", choices=sorted(CONFIGS))
    ap.add_argument("--molecules", type=int, default=0, help="water configs only: override the number of molecules")
    ap.add_argument("--cpu-steps", type=int, default=3, help="steps of the cpu_baseline sample (0 = skip)")
    ap.add_argument("--reduce", default="auto", choices=["auto", "peer", "nccl"],
                    help="multi-GPU reduction of the partial forces: this library's peer-memory kernel or NCCL")
    ap.add_argument("--skin", type=float, default=0.0,
                    help="experiment: Verlet skin (A) of the end-to-end arm; the atoms then move ballistically "
                         "(300 K Maxwell-Boltzmann velocities, 1 fs per step) so that grid reuse is exercised")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of each timed path returned as DIR/<name>.npy (rank 0): "
                         "energies (f64) and grad = dE/dcoords (f32) of the device step, e2e_energies (f64) and "
                         "e2e_forces (f32) of the host-buffer step; the inputs are seeded, so two builds can be "
                         "compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        work = make_workload(args.config, args.molecules)
        n_atoms = work["n_atoms"]
        times, kind, threads, what = run_cpu_reference(work, args.steps, args.warmup, budget_s=240.0)
        t = statistics.median(times)
        value = n_atoms / t
        config = {"workload": CONFIGS[args.config], "name": args.config, "atoms": n_atoms, "conformers": work["n_conf"],
                  "ensemble": 8, "aev_dim": 1008, "cutoffs_A": [5.1, 3.5], "parallelism": f"{threads} CPU threads"}
        sample = (f"{len(times)} full energy+force evaluations of the workload ({n_atoms} atoms), median; {what}; "
                  f"{threads} threads = physical cores of this host")
        line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
                "steps": len(times), "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "ns_per_day": 0.0864 / t, "conformers_per_s": work["n_conf"] / t, "config": config,
                "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
                "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "step_times_s": [round(x, 4) for x in times], "gpu_launches": 0}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ B200 arm
    import torch.distributed as dist
    if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"  # keep stdout to the one JSON line (NCCL prints its version there)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from torchani_b200 import models
    from torchani_b200.calculator import HostCalculator
    from torchani_b200.parallel import ShardedEngine
    from torchani_b200.synthetic import DIMS_2X, make_weights

    work = make_workload(args.config, args.molecules)
    n_atoms, n_conf = work["n_atoms"], work["n_conf"]
    z, idx, coords, cell, pbc = work["z"], work["idx"], work["coords"], work["cell"], work["pbc"]
    periodic = pbc is not None
    weights = make_weights(models.SYMBOLS_2X, DIMS_2X, 1008, 8, seed=1234)
    model = models.from_weight_lists("2x", weights, device=dev, periodic_table_index=True)
    eng = model.engine(dev)
    sharded = ShardedEngine(eng, reduce=args.reduce)
    sp_d, co_d = idx.to(dev), coords.to(dev)
    ce_d = cell.to(dev) if periodic else None
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def one_step():
        return sharded.step(sp_d, co_d, ce_d, periodic)

    sampler = ClockSampler(local_rank)
    sampler.start()  # sampled from the warm-up to the end of the end-to-end region (GPU under load throughout)
    for _ in range(max(warmup, eng.graph_after + 2)):   # eager uses + the graph capture happen here, untimed
        one_step()
    eng.check_status()
    barrier()
    evs = []
    for _ in range(args.steps):
        flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = one_step()
        b.record()
        evs.append((a, b))
    barrier()
    # copied now: the step's result tensors are workspace buffers that later steps overwrite
    dumps = {"energies": out[0].cpu().numpy(), "grad": out[1].cpu().numpy()}
    total_ms = sum(a.elapsed_time(b) for a, b in evs)
    t_all = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_all, op=dist.ReduceOp.MAX)
    ms_per_step = float(t_all.item()) / args.steps
    value = n_atoms / (ms_per_step * 1e-3)
    eng.check_status()
    launches_per_step = eng.launches_per_step + (1 if sharded.mode == "peer" else 0)

    # ---- end to end through the public API with HOST buffers (pinned host inputs -> host energy + forces;
    #      H2D, kernels, multi-GPU reduction, D2H and the synchronisation inside the timed region)
    h_vel = None
    if not work["batch"]:
        calc = HostCalculator(model, z[0].numpy(), cell.numpy() if periodic else None, pbc=periodic,
                              skin=args.skin, sharded=sharded if world > 1 else None)
        h_pos = coords[0].numpy().copy()
        if args.skin > 0:   # A/fs: sqrt(kT/m), kT = 0.02585 eV, 1 amu A^2/fs^2 = 103.6427 eV
            mass = np.where(z[0].numpy() == 1, 1.008, 15.999)[:, None]
            h_vel = (np.random.default_rng(0).normal(size=h_pos.shape) * np.sqrt(0.02585 / (103.6427 * mass))).astype("float32")

        def e2e_step():
            if h_vel is not None:
                h_pos[...] += h_vel
            return calc.calculate(h_pos)

        api = ("torchani_b200.calculator.HostCalculator.calculate (host positions in, host energy+forces out; "
               "counterpart of torchani.ase.Calculator.calculate)")
        h2d, d2h = calc.h2d_bytes, calc.d2h_bytes
        e2e_warm = calc.graph_after + 3
    else:
        # batch of conformers: the model-level call of grad.py:263-290 on pinned host tensors
        h_z = z.pin_memory()
        h_c = coords.pin_memory()
        h_f = torch.empty(coords.shape, dtype=torch.float32).pin_memory()
        h_e = torch.empty(n_conf, dtype=torch.float64).pin_memory()

        def e2e_step():
            zd = h_z.to(dev, non_blocking=True)
            cd = h_c.to(dev, non_blocking=True)
            if world > 1:
                e, g = sharded.step(model.species_converter(zd), cd, None, False)
                f = -g
            else:
                e, f = model.energies_and_forces(zd, cd)
            h_f.copy_(f.to(torch.float32), non_blocking=True)
            h_e.copy_(e, non_blocking=True)
            torch.cuda.current_stream(dev).synchronize()
            return h_e, h_f

        api = "torchani_b200.models.ANI.energies_and_forces on pinned host tensors (grad.py:263-290), results to the host"
        h2d = h_z.numel() * 8 + h_c.numel() * 4
        d2h = h_f.numel() * 4 + h_e.numel() * 8
        e2e_warm = eng.graph_after + 3
    for _ in range(e2e_warm):   # incl. the graph capture of the host-driven step
        e2e_step()
    barrier()
    e2e_evs = []
    for _ in range(args.steps):
        flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        e2e_out = e2e_step()
        b.record()
        e2e_evs.append((a, b))
    barrier()
    dumps["e2e_energies"] = np.array(e2e_out[0], dtype=np.float64).reshape(-1)
    dumps["e2e_forces"] = np.array(e2e_out[1], dtype=np.float32)
    clocks = sampler.stop()
    e2e_ms = sum(a.elapsed_time(b) for a, b in e2e_evs)
    t_e2e = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    e2e_ms_per_step = float(t_e2e.item()) / args.steps
    e2e_value = n_atoms / (e2e_ms_per_step * 1e-3)

    # ---- per-stage device times for the roofline (separate short run, events per C-ABI call)
    eng.profile = True
    for _ in range(5):
        flush.fill_(1)
        one_step()
    stage = eng.stage_times_ms()
    eng.profile = False
    pk = peaks()
    owned = n_atoms / world
    counts = torch.bincount(idx[idx >= 0].flatten(), minlength=7).tolist()
    flops = sum(eng.nets.flops_per_atom(s) * c for s, c in enumerate(counts)) / world
    mlp_s = stage.get("mlp_forward_backward", float("nan")) * 1e-3
    fwd_s = stage.get("aev_forward", float("nan")) * 1e-3
    bwd_s = stage.get("aev_backward", float("nan")) * 1e-3
    from torchani_b200._lib import operand_format
    fmt = operand_format()
    split = ("2 x fp16 split of every (power-of-two scaled) fp32 operand, 3 products" if fmt.parts == 2
             else "3 x bf16 split of every fp32 operand, 6 products")
    traffic = measured_traffic(args.config) if world == 1 else {}
    # what the tensor cores actually execute: layer 1 over the live 32-column AEV blocks only, every product of the
    # operand split counted (3 for 2 x fp16, 6 for 3 x bf16)
    ws_b = eng.workspace(*idx.shape)
    live_cols = 32 * int(ws_b.aev_blocks[0].item())
    products = 3 if fmt.parts == 2 else 6
    executed = sum(2.0 * (live_cols * h1 + h1 * h2 + h2 * h3 + h3) * eng.nets.num_members * 2 * c
                   for (h1, h2, h3), c in zip(eng.nets.dims, counts)) * products / world
    mlp_kernel = ("tc::k_mlp_fused (ani_b200_mlp_step, one data-flow launch)" if getattr(eng, "mlp_fused", False)
                  else "tc::k_gemm_tc x 6 (ani_b200_mlp_forward_backward, chained launches)")
    roofline = {"kernel": f"{mlp_kernel}: ensemble MLP fwd + bwd-to-input, "
                          f"tcgen05 kind::f16 on a {split} (fp32-accurate)",
                "bound": "tensor", "achieved": flops / mlp_s / 1e12, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
                "frac": flops / mlp_s / 1e12 / pk["bf16_tflops"], "traffic": traffic.get("mlp"),
                "algorithmic_flops_per_launch_sequence": flops, "peak_source": pk["source"],
                "live_aev_columns": live_cols, "executed_tensor_flops_per_launch_sequence": executed,
                "executed_tensor_frac": executed / mlp_s / 1e12 / pk["bf16_tflops"],
                "note": "achieved = dense algorithmic FLOPs of SURVEY 8(d) (2 x MACs x 8 members, forward + "
                        "backward-to-input, per atom by element) / device time of the GEMM launches of one step (CUDA "
                        "events on the launch stream); peak = measured dense bf16 rate (= the fp16 rate).  traffic = "
                        "dram bytes of those launches from an ncu --set full capture of THIS library build "
                        "(profiles/traffic.json, keyed by the library hash) or null"}
    roofline_aev = {
        "forward": {"kernel": "k_aev_forward_cta", "bound": "hbm", "achieved": AEV_FWD_BYTES_PER_ATOM * owned / fwd_s / 1e9,
                    "peak": pk["hbm_gbs"], "unit": "GB/s",
                    "frac": AEV_FWD_BYTES_PER_ATOM * owned / fwd_s / 1e9 / pk["hbm_gbs"],
                    "traffic": traffic.get("aev_forward")},
        "backward": {"kernel": "k_aev_backward", "bound": "hbm", "achieved": AEV_BWD_BYTES_PER_ATOM * owned / bwd_s / 1e9,
                     "peak": pk["hbm_gbs"], "unit": "GB/s",
                     "frac": AEV_BWD_BYTES_PER_ATOM * owned / bwd_s / 1e9 / pk["hbm_gbs"],
                     "traffic": traffic.get("aev_backward")},
        "peak_source": pk["source"]}

    # ---- CPU baseline beside it (rank 0, N = 1 only): bounded sample of the same workload, the real reference
    cpu = None
    if rank == 0 and world == 1 and args.cpu_steps > 0:
        times, kind, threads, what = run_cpu_reference(work, args.cpu_steps, 1, budget_s=30.0)
        t = statistics.median(times)
        cpu = {"value": n_atoms / t, "unit": UNIT, "cores": threads, "kind": kind, "ms_per_step": t * 1e3,
               "sample": f"{len(times)} full energy+force evaluations of the same workload ({n_atoms} atoms), median; "
                         f"{what}; {threads} threads = physical cores of this host"}

    if rank == 0:
        config = {"workload": CONFIGS[args.config], "name": args.config, "atoms": n_atoms, "conformers": n_conf,
                  "ensemble": 8, "aev_dim": 1008, "cutoffs_A": [5.1, 3.5],
                  "parallelism": (f"central-atom sharding x{world} + one in-graph {sharded.mode} reduction of the "
                                  "partial forces") if world > 1 else "single GPU",
                  "l2": "256 MiB flush between timed steps (untimed)"}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "ns_per_day": 0.0864 / (ms_per_step * 1e-3), "conformers_per_s": n_conf / (ms_per_step * 1e-3),
                "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": e2e_ms_per_step, "api": api,
                        **({"verlet_skin_A": args.skin, "grid_rebuilds": calc.rebuilds, "steps_redone": calc.redone,
                            "calls": calc._calls} if args.skin > 0 else {})},
                "gpu_launches": launches_per_step * args.steps,
                "operand_format": {"parts": fmt.parts, "bytes_per_element": 2 * fmt.parts},
                "library_sha256_16": library_hash(), "library_build_id": library_build_id(),
                "stage_ms": stage, "roofline": roofline, "roofline_aev": roofline_aev, "cpu_baseline": cpu}
        if args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in dumps.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
