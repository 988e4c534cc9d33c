"""Device time of the matrix-free orbital Hessian against forming it.
    python tools/hessian_operator_bench.py [--out FILE] [workload ...]
(one JSON line per workload on stdout; with --out the whole result, card name and power limit included, as JSON)

For each workload (default: c6h6_ccpvdz_cas66 = N 114 CAS(6,6), synthetic_n256_cas1212 = N 256 CAS(12,12)) one
OrbitalHessian on the class path at a random rotation, then CUDA-event times (median of REPS after a warm-up) of
  * ``matvec`` for blocks of nv = 1, 2, 4, 8, 16 vectors,
  * ``diagonal()``,
  * ``matrix()`` (building H) and ``matrix() @ V`` for the same blocks.
The class buffer (2 nIp^2 + 1 planes of ld^2 doubles) is larger than the L2 cache at both sizes, so every pass
streams it from HBM.  Reported rates: bytes/s = one read of the class buffer per block of at most 8 vectors over
the time; flop/s = the plane products the kernel runs, 2 ld^2 sum_k |P_k| per vector (|P_k| = distinct p of the
coefficient row k, counted here from the RDM structure), over the time.  The two methods' outputs are compared."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from auto_oo_b200 import OO_energy                                               # noqa: E402
from auto_oo_b200.synthetic import CONFIG_SHAPES, SyntheticMol, random_kappa, random_rdms   # noqa: E402

REPS = 25
NVS = [1, 2, 4, 8, 16]
PASS_VECTORS = 8            # vectors per streamed pass (csrc/hessian_operator.cu kHvpMaxVec)


def timed(fn):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(REPS):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), float(np.min(ts))


def plane_counts(one, two, no, na):
    """sum_k |P_k| and sum_k |R_k| over the class rows: distinct p (r) with a non-zero coefficient A_k[p, r]."""
    from oracle import oo_oracle as orc
    ni = no + na
    d1, d2 = orc.full_rdms(one.cpu(), two.cpu(), ni, np.arange(no), np.arange(no, ni))
    A = torch.cat([(d2.permute(0, 2, 1, 3) + d2.permute(0, 3, 1, 2)).reshape(ni, ni, ni * ni).permute(2, 0, 1),
                   d2.reshape(ni, ni, ni * ni).permute(2, 0, 1), d1[None]]) != 0
    return int(A.any(2).sum()), int(A.any(1).sum())


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[torch.cuda.current_device()] if out else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="write the result as JSON to this file")
    ap.add_argument("workloads", nargs="*", default=["c6h6_ccpvdz_cas66", "synthetic_n256_cas1212"])
    args = ap.parse_args()
    workloads = args.workloads
    dev = torch.device("cuda", 0)
    result = {"card": card(), "reps": REPS, "statistic": "median (min) of CUDA-event times, ms", "workloads": []}
    for w in workloads:
        nao, nelec, ncas, nelecas = CONFIG_SHAPES[w]
        mol = SyntheticMol(nao, nelec, seed=11, device=dev, rng_device="cpu")
        oo = OO_energy(mol, ncas, nelecas, oao_mo_coeff=mol.random_oao_mo_coeff, device=dev)
        mol._B = None
        eng = oo.engine
        one, two = (x.to(dev) for x in random_rdms(ncas, nelecas, seed=11))
        kappa = random_kappa(oo.n_kappa, seed=11, batch=1).to(dev)
        H = oo._hessian(oo._mo_integrals(kappa=kappa[0]), one, two, one)
        nk, ld, nIp = eng.nk, eng.ld, eng.nIp
        cls_bytes = (2 * nIp * nIp + 1) * ld * ld * 8
        sum_p, sum_r = plane_counts(one, two, eng.no, eng.na)
        row = {"workload": w, "N": nao, "no": eng.no, "na": eng.na, "n_kappa": nk, "class_buffer_bytes": cls_bytes,
               "sum_k_P_k": sum_p, "sum_k_R_k": sum_r, "matvec": [], "dense": []}
        t_diag = timed(H.diagonal)
        t_build = timed(H.matrix)
        M = H.matrix()
        row["diagonal_ms"] = t_diag
        row["build_ms"] = t_build
        row["diagonal_max_abs_diff"] = float((H.diagonal() - M.diagonal()).abs().max())
        scale = float(M.abs().max())
        for nv in NVS:
            V = torch.empty(nk, nv, dtype=torch.float64, device=dev).uniform_(-1, 1)
            t = timed(lambda: H.matvec(V))
            t_mm = timed(lambda: M @ V)
            passes = -(-nv // PASS_VECTORS)
            flop = 2.0 * ld * ld * sum_p * nv
            row["matvec"].append({"nv": nv, "ms": t, "class_buffer_passes": passes,
                                  "GB_per_s": passes * cls_bytes / (t[0] * 1e-3) / 1e9,
                                  "plane_TFLOP_per_s": flop / (t[0] * 1e-3) / 1e12,
                                  "max_abs_diff_rel_to_Hmax": float((H.matvec(V) - M @ V).abs().max()) / scale})
            row["dense"].append({"nv": nv, "H_at_V_ms": t_mm, "build_plus_H_at_V_ms": t_build[0] + t_mm[0]})
        del M, H
        eng.release_workspaces()
        torch.cuda.empty_cache()
        result["workloads"].append(row)
        print(json.dumps(row), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps({"card": result["card"]}))


if __name__ == "__main__":
    main()
