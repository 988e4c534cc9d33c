"""Newton mode with the formed Hessian (FP64 eigh) against the matrix-free step (Davidson + deflated PCG on products).
    python tools/newton_solver_bench.py [--out FILE] [--reps R] [workload ...]
(one JSON line per workload on stdout; with --out the whole result, card name and power limit included, as JSON)

For each workload (default: c6h6_ccpvdz_cas66 = N 114 CAS(6,6), synthetic_n256_cas1212 = N 256 CAS(12,12)) one
``energy_gradient_newton_direction`` at a seeded random rotation, dense (default) and ``matrix_free=True``:
CUDA-event medians over R runs after a warm-up, the products the solver took (Davidson / CG), the peak device memory
of a call beyond what was allocated before it (after a warm-up call), and max|delta dp|, |delta lambda_0| between the
two.  The evaluation alone (``want_hessian=False``) is timed too, so the solver's share is visible."""
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
from auto_oo_b200 import oo_energy as _oo                                         # noqa: E402
from auto_oo_b200.synthetic import CONFIG_SHAPES, SyntheticMol, random_kappa, random_rdms   # noqa: E402

SEED = 11


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), float(np.min(ts))


def peak_extra(fn):
    fn()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return int(torch.cuda.max_memory_allocated() - base)


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[torch.cuda.current_device()] if out else "unknown"


def run(workload, reps):
    dev = torch.device("cuda", 0)
    nao, nelec, ncas, nelecas = CONFIG_SHAPES[workload]
    mol = SyntheticMol(nao, nelec, seed=SEED, device=dev, rng_device="cpu")
    oo = OO_energy(mol, ncas, nelecas, oao_mo_coeff=mol.random_oao_mo_coeff, device=dev)
    mol._B = None
    eng = oo.engine
    one, two = (x.to(dev) for x in random_rdms(ncas, nelecas, seed=SEED))
    k = random_kappa(oo.n_kappa, seed=SEED, batch=1).to(dev)
    Coao = eng.to_padded(oo.oao_mo_coeff, 2)
    res = {"workload": workload, "nao": nao, "ncas": ncas, "n_kappa": oo.n_kappa, "reps": reps}
    res["evaluation_only_ms"] = timed(lambda: eng.evaluate(Coao, one, two, kappa=k, want_hessian=False,
                                                           path=oo.integral_path), reps)[0]
    dense = oo.energy_gradient_newton_direction(k, one, two)
    res["dense_ms"], res["dense_min_ms"] = timed(lambda: oo.energy_gradient_newton_direction(k, one, two), reps)
    res["dense_peak_extra_mb"] = peak_extra(lambda: oo.energy_gradient_newton_direction(k, one, two)) / 2 ** 20
    eng.release_workspaces()
    torch.cuda.empty_cache()
    # solver statistics of the matrix-free step (the OrbitalHessian.newton_step calls of the driver)
    info = {}
    orig = _oo.OrbitalHessian.newton_step

    def counted(self, gradient, **kw):
        return orig(self, gradient, info=info, **kw)
    _oo.OrbitalHessian.newton_step = counted
    try:
        mf = oo.energy_gradient_newton_direction(k, one, two, matrix_free=True)
    finally:
        _oo.OrbitalHessian.newton_step = orig
    res["mf_ms"], res["mf_min_ms"] = timed(lambda: oo.energy_gradient_newton_direction(k, one, two, matrix_free=True),
                                           reps)
    res["mf_peak_extra_mb"] = peak_extra(lambda: oo.energy_gradient_newton_direction(k, one, two,
                                                                                     matrix_free=True)) / 2 ** 20
    res.update({key: info[key] for key in ("davidson_products", "davidson_iterations", "davidson_restarts",
                                           "cg_products", "shift", "lowest_eigenvalue")})
    res["products"] = info["davidson_products"] + info["cg_products"]
    res["identical_E_G"] = bool(torch.equal(dense[0], mf[0]) and torch.equal(dense[1], mf[1]))
    res["max_abs_ddp"] = (dense[2] - mf[2]).abs().max().item()
    res["max_abs_dp"] = dense[2].abs().max().item()
    res["abs_dlambda0"] = abs(dense[3][0].item() - mf[3][0].item())
    res["speedup"] = res["dense_ms"] / res["mf_ms"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("workloads", nargs="*", default=["c6h6_ccpvdz_cas66", "synthetic_n256_cas1212"])
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("newton_solver_bench needs a CUDA device")
    out = {"device": card(), "timing": "CUDA events, median", "results": []}
    for w in a.workloads:
        r = run(w, a.reps)
        print(json.dumps(r), flush=True)
        out["results"].append(r)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
