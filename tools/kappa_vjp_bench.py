"""Device time of the kappa adjoint: the rotation VJP alone, ``energy_from_kappa`` and forward + ``backward()``.
    python tools/kappa_vjp_bench.py [--out FILE] [workload ...]
(one JSON line per workload on stdout; with --out the whole result, card name and power limit included, as JSON)

For each workload (default: c6h6_ccpvdz_cas66 = N 114 CAS(6,6), synthetic_n256_cas1212 = N 256 CAS(12,12), seeded
``SyntheticMol``, class path) CUDA-event medians over REPS calls after a warm-up of
  * ``HotPathEngine.rotation_vjp`` (one ``oo_kappa_rotation_vjp_f64``) and ``HotPathEngine.rotation`` beside it,
  * ``energy_from_kappa`` at a fresh kappa per call (rotation + class transform + energy: the transform misses the
    integral cache every time),
  * the same forward followed by ``backward()`` on a kappa that requires grad.
The backward is the difference of the last two."""
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

REPS = 20


def timed(fn, reps=REPS):
    fn(-1)
    torch.cuda.synchronize()
    ts = []
    for i in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn(i)
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), float(np.min(ts))


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[torch.cuda.current_device()] if out else "unknown"


def bench(workload):
    dev = torch.device("cuda", 0)
    nao, nelec, ncas, nelecas = CONFIG_SHAPES[workload]
    mol = SyntheticMol(nao, nelec, seed=11, device=dev, rng_device="cpu")
    oo = OO_energy(mol, ncas, nelecas, oao_mo_coeff=mol.random_oao_mo_coeff, device=dev)
    eng = oo.engine
    one, two = (t.to(dev) for t in random_rdms(ncas, nelecas, seed=11))
    kappas = random_kappa(oo.n_kappa, seed=11, scale=0.05, batch=REPS + 1).to(dev)
    Ubar = torch.randn(1, eng.ld, eng.ld, dtype=torch.float64, device=dev)
    res = {"workload": workload, "nao": nao, "ncas": ncas, "n_kappa": oo.n_kappa, "reps": REPS}
    res["rotation_ms"] = timed(lambda i: eng.rotation(kappas[i:i + 1] if i >= 0 else kappas[-1:]))
    res["rotation_vjp_ms"] = timed(lambda i: eng.rotation_vjp(kappas[i:i + 1] if i >= 0 else kappas[-1:], Ubar))
    res["energy_forward_ms"] = timed(lambda i: oo.energy_from_kappa(kappas[i], one, two))

    def fwd_bwd(i):
        k = kappas[i].clone().requires_grad_(True)
        oo.energy_from_kappa(k, one, two).backward()
    res["energy_forward_backward_ms"] = timed(fwd_bwd)
    res["backward_ms_median_difference"] = res["energy_forward_backward_ms"][0] - res["energy_forward_ms"][0]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("workloads", nargs="*", default=["c6h6_ccpvdz_cas66", "synthetic_n256_cas1212"])
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("kappa_vjp_bench needs a CUDA device")
    out = {"card": card(), "timing": "CUDA-event median / min over reps, ms", "results": []}
    for w in a.workloads:
        r = bench(w)
        print(json.dumps(r), flush=True)
        out["results"].append(r)
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
