"""``bench.py --dump-outputs DIR``: the results of the last timed step as float64 .npy files (at most 64 MB) from
inputs that are the same in every run, so that two builds can be compared output for output.  CPU: the Hessian
sample and the ``--steps`` check; GPU: the dump of a real run is that step's E, gradient and Hessian."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("E", "G", "H_diag", "H_sample")


def test_hessian_sample_is_the_same_seeded_positions_in_every_evaluation(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_H_ENTRIES", 64)
    B, nk = 2, 20
    H = torch.arange(nk * nk, dtype=torch.float64).reshape(1, nk, nk) + 1000.0 * torch.arange(B, dtype=torch.float64)[:, None, None]
    E, G = torch.randn(B, dtype=torch.float64), torch.randn(B, nk, dtype=torch.float64)
    bench.dump_outputs(str(tmp_path / "a"), E, G, H)
    bench.dump_outputs(str(tmp_path / "b"), E, G, H)
    d = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in NAMES}
    assert all(a.dtype == np.float64 for a in d.values())
    assert np.array_equal(d["E"], E.numpy()) and np.array_equal(d["G"], G.numpy())
    assert np.array_equal(d["H_diag"], H.diagonal(dim1=1, dim2=2).numpy())
    pos = d["H_sample"] - 1000.0 * np.arange(B)[:, None]        # entry value = flat position + 1000 b
    assert pos.shape == (B, 32) and np.array_equal(pos[0], pos[1])
    assert np.all(np.diff(pos[0]) >= 0) and pos.min() >= 0 and pos.max() < nk * nk
    for n in NAMES:
        assert np.array_equal(d[n], np.load(tmp_path / "b" / f"{n}.npy"))


def test_steps_below_one_is_an_error():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True,
                         text=True, timeout=300)
    assert res.returncode != 0 and "--steps must be at least 1" in res.stderr


@pytest.mark.gpu
def test_dump_is_the_last_timed_step_and_repeats_exactly(tmp_path):
    from auto_oo_b200 import OO_energy
    from auto_oo_b200.synthetic import CONFIG_SHAPES, SyntheticMol, random_rdms, random_kappa
    wl, B, steps, warmup = "n2_ccpvdz_cas66", 4, 2, 3
    dumps = []
    for run in ("a", "b"):
        out = tmp_path / run
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", wl, "--steps", str(steps),
                              "--warmup", str(warmup), "--batch-per-gpu", str(B), "--no-cpu-baseline", "--no-e2e",
                              "--no-full-transform-arm", "--dump-outputs", str(out)],
                             capture_output=True, text=True, timeout=900)
        assert res.returncode == 0, res.stderr[-3000:]
        line = json.loads(res.stdout.strip().splitlines()[-1])
        assert line["steps"] == steps
        assert sum(os.path.getsize(out / f"{n}.npy") for n in NAMES) <= 64 << 20
        dumps.append({n: np.load(out / f"{n}.npy") for n in NAMES})
    for n in NAMES:
        assert dumps[0][n].dtype == np.float64 and np.array_equal(dumps[0][n], dumps[1][n]), n

    # the same step through the public API: bench.py's seeded inputs, the rotations of the last timed step
    nao, nelec, ncas, nelecas = CONFIG_SHAPES[wl]
    dev = torch.device("cuda", 0)
    mol = SyntheticMol(nao, nelec, seed=5, device=dev)
    oo = OO_energy(mol, ncas, nelecas, oao_mo_coeff=mol.random_oao_mo_coeff, device=dev)
    one, two = random_rdms(ncas, nelecas, seed=5, device=dev)
    nk = oo.n_kappa
    kappa = random_kappa(nk, seed=1000, device=dev, batch=(warmup + steps) * B)[-B:]
    E, G, H = (t.cpu().numpy() for t in oo.energy_gradient_hessian(kappa, one, two))
    d = dumps[0]
    assert d["E"].shape == (B,) and d["G"].shape == (B, nk) and d["H_sample"].shape == (B, nk * nk)
    assert np.abs(d["E"] - E).max() < 1e-9 and np.abs(d["G"] - G).max() < 1e-9
    assert np.abs(d["H_diag"] - np.diagonal(H, axis1=1, axis2=2)).max() < 1e-8
    assert np.abs(d["H_sample"] - H.reshape(B, -1)).max() < 1e-8
