#!/usr/bin/env python
"""Benchmark of the orbital-optimization hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME]

One *evaluation* (SURVEY section 8d): given (h, g, S^-1/2, E_nuc, C_oao) resident and a rotation
kappa, gamma, Gamma -> E, the packed orbital gradient (n_kappa) and the Hessian (n_kappa^2) at
C' = S^-1/2 C_oao expm(-K(kappa)).  One *step* = one batch of ``--batch-per-gpu`` evaluations on
every rank (different kappa per evaluation; ranks hold replicas of the integrals and disjoint
kappa sets, no data-path collective => weak scaling).  Default workload: BASELINE config 5,
synthetic N=256 AO basis, CAS(12,12), random symmetric RDMs.

Prints ONE JSON line (rank 0).  Every key describes the SAME timed arm unless its name says otherwise:

* ``value`` / ``ms_per_step``: evaluations/s with all inputs resident in HBM (J/K-class transform path).
* ``roofline``: the dominant kernel group of that arm -- the 7 ``dgemm_tn_kernel`` launches of the class
  transform of every evaluation, timed with CUDA events inside the timed region; ``roofline_kernels``: each of
  the 7 launches timed alone in a separate pass (stage flags of ``oo_class_transform_sym_f64``);
  ``roofline_hbm``: the HBM-bound stages (energy, Fock/gradient, Hessian) of the timed region against the
  measured copy bandwidth of MEASURED_PEAKS.json; ``roofline_full_transform``: the complete four-index
  transform (8 N^5 flop, BASELINE's "4-index FP64 TFLOPS vs peak"), measured in its own arm.
  FP64 peak: cuBLAS DGEMM measured in the same run (MEASURED_PEAKS.json has no FP64 entry; nominal 40 TFLOP/s).
* ``e2e``: the same metric through ``OO_energy.energy_gradient_hessian`` with HOST tensors (pinned H2D of
  kappa/gamma/Gamma, D2H of E, G and the Hessian inside the timed region) in the throughput configuration:
  lower-triangle Hessians, pinned result buffers, two calls in flight; ``e2e_dense``: dense Hessians, one call at a
  time (round-1 behaviour); ``e2e_newton``: Newton mode, the Hessian is consumed on the device.
* ``cpu_baseline`` / ``--impl reference``: the VERBATIM reference (baseline/_ref, loaded behind
  oracle/ref_shim.py) on the host cores: its three calls energy_from_kappa + analytic_gradient +
  analytic_hessian at N = 96 with the workload's CAS, extrapolated to N = 256 by its own flop count (the
  reference cannot run at N = 256: a dozen N^4 tensors); ``cpu_baseline_measured``: a same-config measurement
  of both implementations at the largest BASELINE config the reference can run (114 AOs, CAS(6,6)).  The
  reference is not part of this repository: without it both are null and ``cpu_baseline_unavailable`` says why.

``--dump-outputs DIR`` writes the results of the last timed step as float64 ``DIR/<name>.npy`` (see
``dump_outputs``), so that two builds can be compared on the same seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

F64 = torch.float64
METRIC = "oo_energy_gradient_hessian_evals_per_sec"
UNIT = "evals/s"
# the CPU reference runs the workload's CAS at this basis size whatever --steps / --warmup are (N=256 cannot run
# on a host); one E+G+H sample is 10-15 s on 16 cores.  The budget caps the warm-up repetitions.
CPU_SAMPLE_NAO = int(os.environ.get("OO_BENCH_CPU_SAMPLE_NAO", "96"))
CPU_BUDGET_S = float(os.environ.get("OO_BENCH_CPU_BUDGET_S", "150"))
MEASURED_WORKLOAD = "c6h6_ccpvdz_cas66"           # same-config secondary: the reference can run this one
DUMP_H_ENTRIES = 1 << 22                          # Hessian entries --dump-outputs keeps over the whole batch (32 MB)
DUMP_MAX_BYTES = 64 << 20


# --------------------------------------------------------------------------------------
def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "power_w_max": max(pw),
                "samples": len(sm), "reasons": sorted(reasons)}


def measure_fp64_dgemm_peak(n=8192, reps=5):
    """cuBLAS DGEMM n^3, best of reps (the FP64 denominator; MEASURED_PEAKS.json has none)."""
    a = torch.randn(n, n, dtype=F64, device="cuda")
    b = torch.randn(n, n, dtype=F64, device="cuda")
    c = torch.empty_like(a)
    for _ in range(2):
        torch.matmul(a, b, out=c)
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b, out=c)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) * 1e-3)
    del a, b, c
    torch.cuda.empty_cache()
    return 2 * n ** 3 / best / 1e12


def hbm_peak_gbs():
    """Measured copy bandwidth of this pool's B200s (driver-written), else the profiling recipe's fallback."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except (OSError, KeyError, ValueError):
        return 6553.3, "fallback (MEASURED_PEAKS.json absent): 6553.3 GB/s measured on this pool in round 1"


def dump_outputs(out_dir, E, G, H):
    """Writes one step's results (B evaluations) as float64 ``out_dir/<name>.npy``: ``E`` (B,), the packed gradient
    ``G`` (B, n_kappa), the Hessian diagonal ``H_diag`` (B, n_kappa) and ``H_sample`` (B, S), the Hessian entries at
    S flat positions of the n_kappa x n_kappa matrix drawn once from a fixed seed (the same positions in every
    evaluation and every run; all entries, in order, when they fit DUMP_H_ENTRIES)."""
    import numpy as np
    B, nk = G.shape
    n = min(nk * nk, DUMP_H_ENTRIES // B)
    if n == nk * nk:
        idx = torch.arange(n)
    else:
        idx = torch.randint(nk * nk, (n,), generator=torch.Generator().manual_seed(0)).sort().values
    arrays = {"E": E, "G": G, "H_diag": H.diagonal(dim1=1, dim2=2),
              "H_sample": H.reshape(B, nk * nk)[:, idx.to(H.device)]}
    arrays = {k: v.detach().to("cpu", F64).contiguous().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, f"--dump-outputs would write {total} bytes (limit {DUMP_MAX_BYTES})"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# --------------------------------------------------------------------------------------
# CPU arm: the verbatim reference behind the pennylane.math shim
# --------------------------------------------------------------------------------------
_ref_problems = {}


def reference_problem(shape_name, nao_sample):
    """(reference OO_energy, RDMs, kappa) for the workload's CAS at ``nao_sample`` orbitals (or the workload's
    own basis if smaller); inputs are generated once, outside any timing."""
    from auto_oo_b200.synthetic import CONFIG_SHAPES, SyntheticMol, random_rdms, random_kappa
    from oracle.ref_shim import load_reference
    nao, nelec, ncas, nelecas = CONFIG_SHAPES[shape_name]
    ns = min(nao, nao_sample)
    nelec_s = min(nelec, 2 * (ns - ncas) + nelecas)
    nelec_s -= (nelec_s - nelecas) % 2
    key = (shape_name, ns)
    if key not in _ref_problems:
        ref = load_reference()
        mol = SyntheticMol(ns, nelec_s, seed=5)
        one, two = random_rdms(ncas, nelecas, seed=5)
        oo = ref.oo_energy.OO_energy(mol, ncas, nelecas, oao_mo_coeff=mol.random_oao_mo_coeff,
                                     freeze_active=False, interface='torch')
        _ref_problems[key] = (oo, one, two, random_kappa(oo.n_kappa, seed=5), mol)
    return _ref_problems[key] + (nao, ns)


def reference_evaluation(oo, one, two, kappa):
    """One evaluation the way a user of the reference obtains it (oo_energy.py:199-202, :404-424)."""
    Cp = oo.mo_coeff @ oo.kappa_to_mo_coeff(kappa)
    E = oo.energy_from_kappa(kappa, one, two)
    G = oo.kappa_matrix_to_vector(oo.analytic_gradient(one, two, mo_coeff=Cp))
    H = oo.full_hessian_to_matrix(oo.analytic_hessian(one, two, mo_coeff=Cp))
    return E, G, H


def cpu_reference_sample(shape_name, nao_sample, reps=1):
    """Seconds per reference evaluation at ``nao_sample`` orbitals (best of reps) and the factor that carries
    it to the workload's basis size: the reference's own flop count, three four-index transforms and the dense
    Y-matrix, 3*8N^5 + 6N^6."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    oo, one, two, kappa, _, nao, ns = reference_problem(shape_name, nao_sample)
    best = float("inf")
    for _ in range(reps):
        t0 = time.perf_counter()
        outputs = reference_evaluation(oo, one, two, kappa)
        best = min(best, time.perf_counter() - t0)
    flops = lambda n: 24.0 * n ** 5 + 6.0 * n ** 6
    scale = flops(nao) / flops(ns)
    return {"seconds_sample": best, "nao_sample": ns, "scale": scale, "cores": cores,
            "evals_per_s": 1.0 / (best * scale), "outputs": outputs}


def cpu_baseline_dict(r, nao):
    d = {"value": r["evals_per_s"], "unit": UNIT, "cores": r["cores"], "kind": "reference",
         "extrapolated": r["scale"] != 1.0, "sample_nao": r["nao_sample"], "scale": r["scale"],
         "seconds_sample": r["seconds_sample"],
         "sample": f"verbatim reference (baseline/_ref behind oracle/ref_shim.py, torch {torch.__version__} CPU, "
                   f"{r['cores']} threads): energy_from_kappa + analytic_gradient + analytic_hessian at "
                   f"N={r['nao_sample']} with the workload's CAS took {r['seconds_sample']:.2f} s"}
    if d["extrapolated"]:
        d["sample"] += (f"; scaled to N={nao} by the reference's flop count 24N^5+6N^6 (x{r['scale']:.0f}) -- an "
                        f"extrapolation: the reference cannot run at N={nao} (a dozen N^4 tensors, 400 GB)")
    return d


def run_reference(args, rank, world):
    """--impl reference: the verbatim reference on the host cores (rank 0 only)."""
    if rank != 0:
        return
    from auto_oo_b200.synthetic import CONFIG_SHAPES
    nao, nelec, ncas, nelecas = CONFIG_SHAPES[args.workload]
    first = cpu_reference_sample(args.workload, CPU_SAMPLE_NAO)             # warm-up (also sizes the budget)
    per = first["seconds_sample"]
    for _ in range(min(max(args.warmup, 1) - 1, max(0, int(0.2 * CPU_BUDGET_S / per)))):
        cpu_reference_sample(args.workload, CPU_SAMPLE_NAO)
    # same sample size whatever --steps is; every step is one evaluation of that sample
    measured = args.steps
    wall, res = 0.0, None
    for _ in range(measured):
        res = cpu_reference_sample(args.workload, CPU_SAMPLE_NAO)
        wall += res["seconds_sample"]
    res = dict(res, seconds_sample=wall / measured)
    res["evals_per_s"] = 1.0 / (res["seconds_sample"] * res["scale"])
    value = res["evals_per_s"]
    cpu = cpu_baseline_dict(res, nao)
    cpu["steps_measured"] = measured
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["seconds_sample"] * res["scale"] * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": args.workload, "nao": nao, "cas": [nelecas, ncas]},
        "cpu_baseline": cpu,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if args.dump_outputs:
        E, G, H = (torch.as_tensor(x)[None] for x in res["outputs"])
        dump_outputs(args.dump_outputs, E, G, H)
    print(json.dumps(line), flush=True)


def same_config_measurement(dev):
    """Both implementations on the largest BASELINE config the reference can run (config 4 shape: 114 AOs,
    CAS(6,6), n_kappa = 2283): one reference evaluation on the host cores, and the CUDA path through the public
    host-tensor API on the same inputs; differences of the results are reported alongside."""
    from auto_oo_b200 import OO_energy
    oo_ref, one, two, kappa, mol, nao, ns = reference_problem(MEASURED_WORKLOAD, 10 ** 9)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    t0 = time.perf_counter()
    Er, Gr, Hr = reference_evaluation(oo_ref, one, two, kappa)
    t_ref = time.perf_counter() - t0
    oo = OO_energy(mol, oo_ref.ncas, oo_ref.nelecas, oao_mo_coeff=mol.random_oao_mo_coeff, device=dev)
    kb = kappa[None].repeat(8, 1)
    for _ in range(3):
        oo.energy_gradient_hessian(kb, one, two)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    reps = 5
    for _ in range(reps):
        E, G, H = oo.energy_gradient_hessian(kb, one, two)
    t_ours = (time.perf_counter() - t0) / (reps * kb.shape[0])
    out = {"workload": MEASURED_WORKLOAD, "nao": nao, "n_kappa": int(oo.n_kappa), "extrapolated": False,
           "reference": {"value": 1.0 / t_ref, "unit": UNIT, "seconds_per_eval": t_ref, "cores": cores,
                         "kind": "reference"},
           "ours_host_tensors": {"value": 1.0 / t_ours, "unit": UNIT, "seconds_per_eval": t_ours,
                                 "batch": int(kb.shape[0])},
           "ratio": t_ref / t_ours,
           "max_abs_diff": {"E": abs(E[0].item() - Er.item()), "G": (G[0] - Gr).abs().max().item(),
                            "H": (H[0] - Hr).abs().max().item()}}
    del oo
    torch.cuda.empty_cache()
    return out


def strong_arm(args, mol, ncas, nelecas, dev, world, rank, n_evals, max_over_ranks, barrier):
    """ONE evaluation at a time spread over all ranks (pair-sharded class transform + one NCCL all-reduce of the
    class buffer; E, G, H replicated): evaluations/s of the whole job, stage split and the all-reduce share."""
    from auto_oo_b200 import OO_energy
    from auto_oo_b200.synthetic import random_rdms, random_kappa
    oo = OO_energy(mol, ncas, nelecas, oao_mo_coeff=mol.random_oao_mo_coeff, device=dev, shard="pairs")
    eng = oo.engine
    one, two = random_rdms(ncas, nelecas, seed=5, device=dev)
    Coao = eng.to_padded(oo.oao_mo_coeff, 2)
    nk = oo.n_kappa
    kap = random_kappa(nk, seed=77, device=dev, batch=3 + n_evals)           # the SAME rotations on every rank
    squarings = eng.squarings_for(kap)
    H = torch.empty(1, nk, nk, dtype=F64, device=dev)
    for i in range(3):
        eng.evaluate(Coao, one, two, kappa=kap[i:i + 1], squarings=squarings, H_out=H)
    barrier()
    events, eng.pair_shard.timing = {}, []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(3, 3 + n_evals):
        E, G, _ = eng.evaluate(Coao, one, two, kappa=kap[i:i + 1], squarings=squarings, H_out=H, stage_events=events)
    e1.record()
    barrier()
    t = max_over_ranks(e0.elapsed_time(e1) * 1e-3)
    t_ar = sum(a.elapsed_time(b) for a, b in eng.pair_shard.timing) * 1e-3
    chk = torch.stack([E[0], G.abs().sum(), H.diagonal(dim1=1, dim2=2).sum()])
    lo, hi = chk.clone(), chk.clone()
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    sh = eng.pair_shard
    out = {"value": n_evals / t, "unit": UNIT, "ms_per_evaluation": t / n_evals * 1e3, "evaluations": n_evals,
           "n_gpus": world, "scaling": "strong",
           "stage_ms_per_evaluation": {k: sum(a.elapsed_time(b) for a, b in v) / n_evals for k, v in events.items()},
           "allreduce_ms_per_evaluation": t_ar / n_evals * 1e3,
           "allreduce_bytes": int(eng.class_rows() * eng.ld * eng.ld * 8),
           "slab": {"pair_columns": [int(sh.pq_lo), int(sh.pq_lo + sh.pq_cnt)],
                    "eri_bytes_per_gpu": int(eng.packed_eri().numel() * 8)},
           "replicas_agree": bool(((hi - lo).abs() <= 1e-9 * (1 + hi.abs())).all().item()),
           "what": "OO_energy(shard='pairs'): quarter 1 + Coulomb quarter 2 on this rank's pair columns of the 8-fold "
                   "packed integrals, one NCCL all-reduce of the class buffer, E/G/H on every rank"}
    checks = (E[0].item(), G[0].clone(), H[0].diagonal().sum().item())
    del oo, eng
    torch.cuda.empty_cache()
    return out, checks, (E, G, H)


# --------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="synthetic_n256_cas1212")
    ap.add_argument("--batch-per-gpu", type=int, default=4)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-full-transform-arm", action="store_true")
    ap.add_argument("--mode", default="weak", choices=["weak", "strong"],
                    help="weak: every GPU evaluates its own rotations (replicas; the headline metric).  strong: "
                         "every evaluation is spread over all GPUs (OO_energy(shard='pairs')); with --mode weak and "
                         "N > 1 a short strong-mode arm is reported as well under `strong_scaling`")
    ap.add_argument("--strong-evals", type=int, default=6)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's E, gradient, Hessian diagonal and a seeded "
                         "sample of Hessian entries as float64 DIR/<name>.npy (rank 0; at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3                                   # timing rule: W >= 3
    rank, world, local = dist_env()
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch.distributed as dist
    from auto_oo_b200 import OO_energy, _lib
    from auto_oo_b200.synthetic import CONFIG_SHAPES, SyntheticMol, random_rdms, random_kappa

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_cpus = None
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"               # the version banner goes to stdout, next to the JSON line
        from auto_oo_b200.distributed import bind_to_gpu_numa_node
        visible = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(visible.split(",")[local]) if visible and visible.split(",")[local].isdigit() else local
        numa_cpus = bind_to_gpu_numa_node(phys)                # pinned staging buffers on the GPU's own node
        # NCCL writes its version banner to fd 1 when the communicator is created: keep stdout for the JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    lib = _lib.load()

    nao, nelec, ncas, nelecas = CONFIG_SHAPES[args.workload]
    B = args.batch_per_gpu

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(seconds):
        t = torch.tensor([seconds], dtype=F64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    if args.mode == "strong":
        # ---- only the sharded evaluation: the N^4 tensor is never formed, every rank builds its slab from the
        #      density-fitting factor (this is the mode for bases whose integrals exceed one GPU)
        mol = SyntheticMol(nao, nelec, seed=5, device=dev, build_eri=False)
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        launches0 = lib.oo_launch_count()
        strong, _, last = strong_arm(args, mol, ncas, nelecas, dev, world, rank, args.steps * B, max_over_ranks,
                                     barrier)
        launches = lib.oo_launch_count() - launches0
        clocks = sampler.stop() if rank == 0 else None
        if rank == 0 and args.dump_outputs:
            dump_outputs(args.dump_outputs, *last)
        if rank == 0:
            line = {"metric": METRIC, "value": strong["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
                    "warmup": 3, "ms_per_step": strong["ms_per_evaluation"] * B, "higher_is_better": True,
                    "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                    "config": {"workload": args.workload, "nao": nao, "cas": [nelecas, ncas],
                               "evals_per_step": B, "mode": strong["what"]},
                    "gpu_launches": int(launches), "clocks": clocks, "strong_scaling": strong, "e2e": None,
                    "roofline": None, "cpu_baseline": None}
            print(json.dumps(line), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- synthetic inputs, generated on the device from a fixed seed (every rank: same integrals)
    mol = SyntheticMol(nao, nelec, seed=5, device=dev)
    oo = OO_energy(mol, ncas, nelecas, oao_mo_coeff=mol.random_oao_mo_coeff, device=dev)
    mol._int2e = None                                      # the engine holds the only N^4 copy now
    want_strong = world > 1 or args.mode == "strong"
    if not want_strong:
        mol._B = None                                      # (the strong arm builds its slab from the factor)
    torch.cuda.empty_cache()
    eng = oo.engine
    one, two = random_rdms(ncas, nelecas, seed=5, device=dev)
    Coao = eng.to_padded(oo.oao_mo_coeff, 2)
    nk = oo.n_kappa
    no, na = eng.no, eng.na
    total_steps = args.warmup + args.steps
    # distinct rotations for every rank / step / batch slot
    kappas = random_kappa(nk, seed=1000 + rank, device=dev, batch=total_steps * B).reshape(total_steps, B, nk)
    squarings = eng.squarings_for(kappas.reshape(-1, nk))   # host decision made once, outside the timed region
    H_out = torch.empty(B, nk, nk, dtype=F64, device=dev)

    peak_tf = measure_fp64_dgemm_peak() if rank == 0 else 0.0

    def stage_seconds(events, name):
        return sum(a.elapsed_time(b) for a, b in events.get(name, [])) * 1e-3

    # ---- complete four-index transform arm (the reference's formulation, BASELINE's transform TFLOP/s) ---------
    full_arm = None
    if not args.no_full_transform_arm:
        full_events = {}
        for s in range(args.warmup):
            eng.evaluate(Coao, one, two, kappa=kappas[s], squarings=squarings, H_out=H_out, path="full")
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for s in range(args.warmup, total_steps):
            E_full, G_full, H = eng.evaluate(Coao, one, two, kappa=kappas[s], squarings=squarings, H_out=H_out,
                                             stage_events=full_events, path="full")
        e1.record()
        barrier()
        t_full_local = e0.elapsed_time(e1) * 1e-3
        t_full = max_over_ranks(t_full_local)
        t_transform = stage_seconds(full_events, "transform")
        n_transforms = len(full_events["transform"])
        full_arm = {"E": E_full.clone(), "G": G_full.clone(), "h_diag": H.diagonal(dim1=1, dim2=2).sum().item(),
                    "t": t_full, "t_local": t_full_local, "t_transform": t_transform, "n": n_transforms}
    oo.int2e_ao = None
    eng.drop_full_eri()                                   # keep only the class path's copy of the AO integrals
    torch.cuda.empty_cache()

    # ---- timed arm: device-resident, partial (J/K class) transform ----------------------------------------------
    for s in range(args.warmup):
        eng.evaluate(Coao, one, two, kappa=kappas[s], squarings=squarings, H_out=H_out)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = lib.oo_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    events = {}
    e0.record()
    for s in range(args.warmup, total_steps):
        E, G, H = eng.evaluate(Coao, one, two, kappa=kappas[s], squarings=squarings, H_out=H_out,
                               stage_events=events)
    e1.record()
    barrier()
    launches = lib.oo_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    t_local = e0.elapsed_time(e1) * 1e-3
    t_dev = max_over_ranks(t_local)
    checksum = float(E.sum().item() + G.abs().sum().item() + H.diagonal(dim1=1, dim2=2).sum().item())
    E_dev_last, G_dev_last, H_dev_last = E.clone(), G.clone(), H[-1].clone()
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, E, G, H)
    if full_arm is not None:                              # both formulations must agree on the last step's results
        assert (E - full_arm["E"]).abs().max().item() < 1e-9 and (G - full_arm["G"]).abs().max().item() < 1e-8
        assert abs(H.diagonal(dim1=1, dim2=2).sum().item() - full_arm["h_diag"]) < 1e-6

    # ---- each GEMM launch of the class transform alone (outside the timed region) -------------------------------
    kernel_rows = []
    symmetric = eng.eri_is_symmetric()
    ld, nIp = eng.ld, eng.nIp
    if rank == 0 and symmetric:
        ldp, npIp = int(lib.oo_pair_ld(ld)), int(lib.oo_pair_ld(nIp))
        npair, npI = nao * (nao + 1) // 2, (no + na) * (no + na + 1) // 2
        nI = no + na
        # needed flop per launch: the class index unpadded, quarter 2 over the class pairs n <= m it keeps, the
        # Coulomb quarter 4 over b <= a (J[mn][a][b] is symmetric; the kernel skips the tiles above the diagonal)
        stage_flop = [2.0 * nao * npair * nI * nao,               # quarter 1 over packed AO pairs
                      2.0 * npair * npI * nao,                    # Coulomb quarter 2 (class pairs n <= m)
                      2.0 * nao * npI * nao * nao, 2.0 * npI * nao * npair,
                      2.0 * nao * nao * npI * nao,                # exchange quarter 2 (class pairs n <= m)
                      2.0 * nao * npI * nao * nao, 2.0 * npI * nao * nao * nao]
        names = ["dgemm_tn_kernel Q1 (8-fold packed A rows gathered by bulk copies; pair-unpack epilogue)",
                 "dgemm_tn_tri_kernel J-Q2 (class pairs n <= m)", "dgemm_tn_kernel J-Q3",
                 "dgemm_tn_kernel J-Q4 (b <= a tiles, staged class-expand epilogue)",
                 "dgemm_tn_tri_kernel K-Q2 (class pairs n <= m)",
                 "dgemm_tn_kernel K-Q3", "dgemm_tn_kernel K-Q4 (staged class-expand epilogue)"]
        # (two evaluations per launch where quarter 1 runs on pairs, as in the timed arm; times are per evaluation)
        nst = 2 if (B >= 2 and eng.class_chunk(B) >= 2 and eng.pairs_quarter_one()) else 1
        if nst == 2:
            names[0] = ("dgemm_tn_kernel Q1 (two evaluations side by side: 2 nI columns; 8-fold packed A rows gathered "
                        "by bulk copies; pair-unpack epilogue)")
        Cst = eng.mo_coeff(Coao, eng.rotation(kappas[0, :nst], squarings))
        cbuf = eng.class_integrals(Cst)                    # complete call: every intermediate is in the workspace
        for k in range(7):
            eng.flags = 1 << (16 + k)
            eng.class_integrals(Cst, out=cbuf)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 3
            a.record()
            for _ in range(reps):
                eng.class_integrals(Cst, out=cbuf)
            b.record()
            torch.cuda.synchronize()
            ms = a.elapsed_time(b) / reps / nst            # includes the 18 us h' = C^T h C that rides along
            kernel_rows.append({"kernel": names[k], "algorithmic_flop": stage_flop[k], "ms": ms,
                                "achieved": stage_flop[k] / (ms * 1e-3) / 1e12, "unit": "TFLOP/s",
                                "frac": stage_flop[k] / (ms * 1e-3) / 1e12 / peak_tf})
        eng.flags = 0
        del cbuf

    # ---- end-to-end arms: public API, host tensors in and out -----------------------------------------------------
    e2e = e2e_dense = e2e_newton = None
    if not args.no_e2e:
        kap_host = kappas.cpu()
        one_h, two_h = one.cpu(), two.cpu()
        h2d = 8 * (B * nk + one_h.numel() + two_h.numel())
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

        # (1) throughput configuration: lower-triangle Hessians, pinned results, two calls in flight
        kw = dict(hessian_format="packed", pinned_results=True)
        for s in range(2):
            oo.energy_gradient_hessian(kap_host[s], one_h, two_h, **kw)
        barrier()
        ev0.record()
        pending, sink = None, 0.0
        for s in range(args.warmup, total_steps):
            nxt = oo.energy_gradient_hessian(kap_host[s], one_h, two_h, wait=False, **kw)
            if pending is not None:
                Eh, Gh, Hh = pending.wait()
                sink += float(Eh[0]) + float(Hh[0, 0])     # the results are on the host: read them
            pending = nxt
        Eh, Gh, Hh = pending.wait()
        sink += float(Eh[0]) + float(Hh[0, 0])
        ev1.record()
        barrier()
        t = max_over_ranks(ev0.elapsed_time(ev1) * 1e-3)
        e2e = {"value": world * B * args.steps / t, "unit": UNIT, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": 8 * (B + B * nk + B * nk * (nk + 1) // 2),
               "mode": "hessian_format='packed' (lower triangle of the symmetric Hessian), pinned_results=True, "
                       "wait=False with two calls in flight; every result is read on the host inside the timed region"}
        # the last step's results against the device-resident arm
        assert abs(Eh[-1].item() - E_dev_last[-1].item()) < 1e-9 and (Gh[-1].to(dev) - G_dev_last[-1]).abs().max().item() < 1e-9
        rows_i, cols_i = torch.tril_indices(nk, nk, device=dev)
        assert torch.equal(Hh[-1].to(dev), H_dev_last[rows_i, cols_i])
        del rows_i, cols_i

        # (2) round-1 configuration: dense Hessians, one call at a time (results = views of pinned buffers)
        for s in range(2):
            oo.energy_gradient_hessian(kap_host[s], one_h, two_h, pinned_results=True)
        barrier()
        ev0.record()
        for s in range(args.warmup, total_steps):
            Eh, Gh, Hh = oo.energy_gradient_hessian(kap_host[s], one_h, two_h, pinned_results=True)
        ev1.record()
        barrier()
        t = max_over_ranks(ev0.elapsed_time(ev1) * 1e-3)
        e2e_dense = {"value": world * B * args.steps / t, "unit": UNIT, "h2d_bytes_per_step": h2d,
                     "d2h_bytes_per_step": 8 * (B + B * nk + B * nk * nk),
                     "mode": "hessian_format='dense', pinned_results=True, one call at a time"}
        assert abs(Eh[-1].item() - E_dev_last[-1].item()) < 1e-9
        eng._ws.pop(("slot", 0), None), eng._ws.pop(("slot", 1), None)      # 6 GB of pinned staging memory

        # (3) Newton mode: the Hessian is consumed on the device (eigh + augmented-Hessian shift), only
        #     E, G, the Newton direction and the lowest eigenvalue come back
        nb = 1
        oo.energy_gradient_newton_direction(kap_host[0, :nb], one_h, two_h)
        barrier()
        ev0.record()
        En, Gn, dkn, lamn = oo.energy_gradient_newton_direction(kap_host[args.warmup, :nb], one_h, two_h)
        ev1.record()
        barrier()
        t = max_over_ranks(ev0.elapsed_time(ev1) * 1e-3)
        e2e_newton = {"value": world * nb / t, "unit": UNIT, "h2d_bytes_per_step": 8 * (nb * nk + one_h.numel() + two_h.numel()),
                      "d2h_bytes_per_step": 8 * (2 * nb + 2 * nb * nk), "evaluations": nb,
                      "mode": "energy_gradient_newton_direction: E, G, dkappa = -(H + shift)^-1 G and lambda_0 back; "
                              "the time is dominated by the FP64 eigh of the n_kappa^2 Hessian (cuSOLVER via torch)"}

    # ---- strong-scaling arm: every evaluation spread over all ranks ---------------------------------------------
    strong = None
    if want_strong:
        eng.release_workspaces()
        torch.cuda.empty_cache()
        strong, chk, _ = strong_arm(args, mol, ncas, nelecas, dev, world, rank, args.strong_evals, max_over_ranks,
                                    barrier)
        strong["one_gpu_ms_per_evaluation_same_run"] = t_dev / (B * args.steps) * 1e3
        strong["speedup_vs_one_gpu"] = strong["one_gpu_ms_per_evaluation_same_run"] / strong["ms_per_evaluation"]
        mol._B = None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- rooflines ---------------------------------------------------------------------------------------------
    n_evals = B * args.steps
    t_cls = stage_seconds(events, "transform")
    if symmetric:
        ldp, npIp = int(lib.oo_pair_ld(ld)), int(lib.oo_pair_ld(nIp))
        # needed flop of the seven launches: quarter 1 over packed AO pairs, quarter 2 over the class pairs n <= m
        # (the triangular kernel computes nothing else), two quarters each on the packed class pairs
        cls_flop = (2.0 * ld * ldp * nIp * ld + 2.0 * ldp * npIp * ld + 2.0 * ld * ld * npIp * ld + 6.0 * ld ** 3 * npIp
                    + 2.0 * npIp * ld * ldp)                     # last term: Coulomb quarter 4 over b <= a
        # round 1 counted quarter 2 over ALL class pairs (m, n) -- what its rectangular GEMM executed
        cls_flop_r01 = (2.0 * ld * ldp * nIp * ld + 2.0 * ldp * nIp * nIp * ld + 2.0 * ld * ld * nIp * nIp * ld
                        + 8.0 * ld ** 3 * npIp)
    else:
        cls_flop = cls_flop_r01 = 2.0 * ld ** 4 * nIp + 12.0 * ld ** 3 * nIp * nIp
    traffic = None
    prof = os.path.join(ROOT, "profiles", "class_transform_traffic.json")
    if os.path.exists(prof):
        with open(prof) as f:
            traffic = json.load(f).get(args.workload)
    roofline = {"bound": "tensor",
                "kernel": "dgemm_tn_kernel x5 + dgemm_tn_tri_kernel x2 (J/K-class transform of one evaluation: quarter 1 "
                          "over 8-fold packed AO integrals, three quarters each for the Coulomb and exchange classes; "
                          "FP64 DMMA)",
                "achieved": cls_flop * n_evals / t_cls / 1e12, "peak": peak_tf, "unit": "TFLOP/s",
                "frac": cls_flop * n_evals / t_cls / 1e12 / peak_tf, "traffic": traffic,
                "flop_per_unit": cls_flop,
                "unit_of_work": "one class transform (7 GEMM launches per group of evaluations_per_launch evaluations)",
                "evaluations_per_launch": n_evals // max(1, len(events.get("transform", []))),
                "launch_ms": t_cls / n_evals * 1e3, "launches_timed": 7 * len(events.get("transform", [])),
                "share_of_step": t_cls / t_local,
                "measured_on": "the timed arm (CUDA events on the launching stream around the 7 GEMM launches of every "
                               "group of evaluations, inside the timed region)",
                "peak_source": "cuBLAS FP64 DGEMM 8192^3 measured in this run (MEASURED_PEAKS.json has no FP64 entry); "
                               "nominal B200 FP64 40 TFLOP/s => frac_of_nominal_40tf",
                "frac_of_nominal_40tf": cls_flop * n_evals / t_cls / 1e12 / 40.0,
                "frac_with_round1_flop_count": cls_flop_r01 * n_evals / t_cls / 1e12 / peak_tf,
                "note": "flop = what the seven launches NEED (class index padded to even only, not to the 8-wide MMA "
                        "tile; quarter 2 over class pairs n <= m; Coulomb quarter 4 over b <= a); round 1 counted both "
                        "over everything its rectangular GEMMs executed (frac_with_round1_flop_count, for comparison "
                        "with its 0.835); launch_ms is per class transform"}
    hbm_peak, hbm_src = hbm_peak_gbs()
    N = nao
    nI = no + na
    hbm_bytes = {
        "energy": 8.0 * (2 * no * no + 2 * na * na * no + 2 * na ** 4),
        "fock_gradient": 8.0 * (2 * N * N * no + 2 * N * N * na * na + N * na ** 3 + na ** 4 + 3 * N * N),
        "hessian": 8.0 * ((2 * nI * nI + 1) * N * N + 2 * nI * nI * N * N + nk * nk),
    }
    hbm_kernels = {
        "energy": "active_hamiltonian_kernel + energy_kernel (active_space.py:147-174, oo_energy.py:194-197)",
        "fock_gradient": "fock_core_active_class_kernel + fock_general_kernel + gradient kernels (oo_energy.py:238-309)",
        "hessian": "class Hessian: operand builders, C-block DGEMM, hess_group_stream, hess_spmm, assembly "
                   "(oo_energy.py:311-402); bytes = class buffer once + T written and read + n_kappa^2 out",
    }
    roofline_hbm = []
    for name in ("energy", "fock_gradient", "hessian"):
        t = stage_seconds(events, name)
        if t > 0:
            gbs = hbm_bytes[name] * n_evals / t / 1e9
            roofline_hbm.append({"bound": "hbm", "stage": name, "kernel": hbm_kernels[name], "achieved": gbs,
                                 "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                                 "bytes_per_evaluation": hbm_bytes[name], "ms_per_evaluation": t / n_evals * 1e3,
                                 "share_of_step": t / t_local, "peak_source": hbm_src})
    stage_ms = {k: stage_seconds(events, k) / n_evals * 1e3 for k in events}

    roofline_full = None
    if full_arm is not None:
        ach = 8.0 * nao ** 5 * full_arm["n"] / full_arm["t_transform"] / 1e12
        roofline_full = {"bound": "tensor", "kernel": "dgemm_tn_kernel x4 (complete four-index transform, 2 N^5 flop per "
                                                      "quarter launch)",
                         "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
                         "frac_of_nominal_40tf": ach / 40.0, "flop_per_launch": 2.0 * nao ** 5,
                         "launch_ms": full_arm["t_transform"] / (4 * full_arm["n"]) * 1e3,
                         "share_of_its_step": full_arm["t_transform"] / full_arm["t_local"],
                         "evals_per_s": world * n_evals / full_arm["t"],
                         "measured_on": "its own arm (path='full'), not the arm that produces `value`"}

    from oracle.ref_shim import reference_available
    cpu = cpu_measured = cpu_unavailable = None
    if not args.no_cpu_baseline and not reference_available():
        cpu_unavailable = ("not measured: the auto_oo reference sources are not installed (AUTO_OO_REFERENCE, or "
                           "baseline/_ref; see oracle/ref_shim.py)")
    elif not args.no_cpu_baseline:
        cpu_reference_sample(args.workload, CPU_SAMPLE_NAO)                # warm-up (thread pool, allocator)
        cpu = cpu_baseline_dict(cpu_reference_sample(args.workload, CPU_SAMPLE_NAO, reps=2), nao)   # best of two
        if args.workload == "synthetic_n256_cas1212":
            eng.release_workspaces()
            torch.cuda.empty_cache()
            cpu_measured = same_config_measurement(dev)

    line = {
        "metric": METRIC, "value": world * n_evals / t_dev, "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_dev / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": args.workload, "nao": nao, "cas": [nelecas, ncas], "n_kappa": nk,
                   "evals_per_step_per_gpu": B,
                   "numa_bound_cpus": None if numa_cpus is None else len(numa_cpus),
                   "transform": ("symmetric J/K-class transform (packed AO pairs: N^4 nI + ~7 N^3 nI^2 flop), same E/G/H"
                                 if symmetric else
                                 "general J/K-class transform (2N^4 nI + 12 N^3 nI^2 flop), same E/G/H"),
                   "eri_symmetry_defect": eng.eri_defect,
                   "l2": "inputs larger than L2 (N^4 tensors of %.1f GB)" % (nao ** 4 * 8 / 1e9)
                   if nao ** 4 * 8 > 126e6 else "inputs fit L2; distinct kappa every evaluation"},
        "e2e": e2e, "e2e_dense": e2e_dense, "e2e_newton": e2e_newton, "strong_scaling": strong,
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "roofline_kernels": kernel_rows,
        "roofline_hbm": roofline_hbm, "roofline_full_transform": roofline_full, "stage_ms_per_evaluation": stage_ms,
        "cpu_baseline": cpu, "cpu_baseline_measured": cpu_measured, "cpu_baseline_unavailable": cpu_unavailable,
        "transform_tflops": None if roofline_full is None else roofline_full["achieved"],
        "checksum": checksum,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
