"""bench.py contract on the CPU side: the reference arm (`--impl reference`) needs no GPU, prints ONE JSON line with the
keys the driver reads, and never touches /root/reference at run time."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args, env=None):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args), cwd=ROOT, env=env,
                          stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)


def test_arguments_the_bench_cannot_honour_are_refused():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    for args in (["--impl", "reference", "--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"],
                 ["--workload", "cfg5", "--dump-outputs", "out"]):
        out = _bench(*args, env=env)
        assert out.returncode == 2 and out.stdout == "", args
        assert ("--steps" if "--steps" in args else "--dump-outputs") in out.stderr, args


def test_dump_outputs_keeps_the_same_seeded_rows_of_every_array_above_the_cap(tmp_path, monkeypatch):
    import torch
    import bench
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 20000)
    idx = torch.arange(1000, dtype=torch.float64)[:, None]
    outputs = {"a": idx.expand(-1, 3).contiguous(), "b": idx.expand(-1, 2).float().contiguous()}
    for d in ("one", "two"):
        bench.dump_outputs(str(tmp_path / d), outputs)
    a, b = (np.load(str(tmp_path / "one" / (k + ".npy"))) for k in ("a", "b"))
    assert a.dtype == np.float64 and b.dtype == np.float32 and a.shape[1:] == (3,) and b.shape[1:] == (2,)
    assert sum(os.path.getsize(str(tmp_path / "one" / (k + ".npy"))) for k in ("a", "b")) <= 20000
    rows = a[:, 0]
    assert 0 < rows.size < 1000 and np.all(np.diff(rows) > 0) and np.all(a == rows[:, None]) and np.all(b == rows[:, None])
    assert np.array_equal(np.load(str(tmp_path / "two" / "a.npy")), a)


@pytest.mark.gpu
def test_dump_outputs_writes_the_last_timed_step(tmp_path):
    """--dump-outputs: u, dL/dlogX and the VO residual of the timed step, checked against the CPU oracle like smoke()."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import gpde_b200  # noqa: F401
    from gpde_b200.workloads import Workload
    from oracle import fem_p1, rom_ref, vo_ref
    out = _bench("--workload", "cfg1", "--steps", "3", "--warmup", "1", "--no-sub", "--no-e2e", "--no-cpu-baseline",
                 "--dump-outputs", str(tmp_path))
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout)["steps"] == 3
    got = {k: np.load(os.path.join(str(tmp_path), k + ".npy")) for k in ("u", "grad_logX", "vo_residual")}
    w = Workload("cfg1", seed=0)
    assert got["u"].shape == (w.B, w.n) and got["grad_logX"].shape == (w.B, w.E) and got["vo_residual"].shape == (w.B, w.m)
    assert all(a.dtype == np.float64 for a in got.values())
    P = fem_p1.build_problem(4, 4, 3)
    u0, gX0, _ = rom_ref.rom_fwd_adjoint(torch.tensor(P['M']), torch.tensor(P['bc_dofs_rom']), torch.tensor(w.logX),
                                         torch.tensor(w.F), torch.tensor(w.gbar_u))
    assert np.abs(got["u"] - u0.numpy()).max() < 1e-10 * np.abs(u0.numpy()).max()
    assert np.abs(got["grad_logX"] - gX0.numpy()).max() < 1e-10 * np.abs(gX0.numpy()).max()
    for b in (0, w.B - 1):
        X_DG = fem_p1.image_to_function(w.log_image[b:b + 1].reshape(1, 32, 32), P['pixel_of_cell_fom'])[0]
        K, f = fem_p1.assemble_system_free(P['coords_fom'], P['cells_fom'], np.exp(X_DG), P['bc_dofs_fom'],
                                           w.g_fom[b], P['free_dofs_fom'])
        r0 = vo_ref.vo_residual(K, f, w.V, w.y[b])
        assert np.abs(got["vo_residual"][b] - r0).max() < 1e-10 * np.abs(r0).max()


def test_reference_arm_prints_the_contract_line():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--batch", "128"], cwd=ROOT, env=env, stdout=subprocess.PIPE,
                         stderr=subprocess.PIPE, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    rec = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert key in rec, key
    assert rec["impl"] == "reference" and rec["higher_is_better"] is True and rec["vs_baseline"] is None
    assert rec["config"]["workload"] == "cfg2" and rec["dtype"] == "f64" and rec["data"] == "synthetic"
    assert rec["cpu_baseline"]["kind"] in ("port", "reference") and rec["cpu_baseline"]["cores"] >= 1
    assert rec["e2e"]["h2d_bytes_per_step"] == 0 and rec["e2e"]["d2h_bytes_per_step"] == 0
    assert rec["e2e"]["value"] == rec["value"] and rec["value"] > 0


def test_nothing_reads_the_reference_tree_at_run_time():
    """/root/reference does not exist on the GPU box: the product package, bench.py and the entry points must not
    mention it (only the oracle shim and the golden generator, which run in the build container, do)."""
    offenders = []
    for base, _, files in os.walk(ROOT):
        if any(part in base for part in (".git", "gpurun_out", "__pycache__", os.path.join("tests", "golden"), "build")):
            continue
        for f in files:
            if not f.endswith((".py", ".cu", ".cuh", ".h")):
                continue
            path = os.path.join(base, f)
            rel = os.path.relpath(path, ROOT)
            if rel in (os.path.join("oracle", "ref_shim.py"), os.path.join("tests", "test_bench_contract.py")):
                continue
            if "/root/reference" in open(path, errors="ignore").read():
                offenders.append(rel)
    assert offenders == [], offenders
