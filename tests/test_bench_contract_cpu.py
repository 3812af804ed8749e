"""CPU: the parts of bench.py's contract that do not need a GPU -- the reference arm (`--impl reference`) prints exactly
one JSON line with the required keys, uses all host threads even when a launcher exported OMP_NUM_THREADS=1, and under
a multi-rank launch only rank 0 prints."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env):
    env = dict(os.environ, **extra_env)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "c1", "--steps", "1",
                        "--warmup", "1"], env=env, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    return r.stdout


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    out = _run({"OMP_NUM_THREADS": "1"})  # what torchrun exports to every rank
    lines = [ln for ln in out.splitlines() if ln.strip()]
    assert len(lines) == 1, out
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "cpu_baseline"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "images/s" and d["higher_is_better"] is True and d["value"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == d["value"] and "sample" in cb
    sys.path.insert(0, ROOT)
    import bench
    assert cb["cores"] == bench.usable_cores()  # every core this process may use, not the launcher's OMP_NUM_THREADS=1
    # the sample is a function of the arguments only (same command => same work on every box)
    assert cb["sample"].startswith("1 image = full 256x256 config-c1")
    assert d["config"] == bench.bench_config("c1", 10000, 256, 256, 1)  # the GPU arm prints the same `config`
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and "workload" in d["config"]


def test_reference_arm_is_silent_on_other_ranks():
    out = _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert out.strip() == ""


def test_cpu_baseline_imports_survive_the_reference_gpu_helpers():
    """bench.py's default run measures `ref_gpu` (flat helper modules under oracle/, which put that directory on
    sys.path) and then `cpu_baseline` (the package `oracle`) in ONE process: the second import must still find the
    package.  (Rounds-2 bench lines r2u / r2y carried cpu_baseline None because it did not.)"""
    import subprocess
    import sys

    code = ("import sys; sys.argv=['bench.py']; import bench; bench.import_oracle_helpers(); "
            "step, d = bench.cpu_step_factory('c1'); from oracle import oracle as O; "
            "assert hasattr(sys.modules['oracle'], '__path__'); print('ok', O.__name__)")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ok oracle.oracle" in r.stdout, r.stderr[-800:]


def _stand_in_model(n, layout):
    """The parameter shapes of gsplat.dp.FlatGaussians (SH degree 3, 16 camera rows) over one flat buffer; every row of
    every per-Gaussian parameter starts with its Gaussian's index."""
    import types

    import torch

    widths = dict(means=3, log_scales=3, quats=4, opacity_logit=1)
    widths.update(sh=48) if layout == "block" else widths.update(sh_dc=3, sh_rest=45)
    flat = torch.zeros(n * sum(widths.values()))
    params, off = {}, 0
    for name, w in widths.items():
        params[name] = flat[off:off + n * w].view(n, w)
        params[name][:, 0] = torch.arange(n, dtype=torch.float32)
        off += n * w
    return types.SimpleNamespace(N=n, flat=flat, params=params, cam_vel=torch.ones(16, 6))


def test_dump_outputs_stays_under_64_mb_with_the_same_rows(tmp_path):
    """bench.py --dump-outputs at the largest configs (c5: 2M Gaussians): every per-Gaussian parameter is written for one
    seeded set of rows, the loss and the camera velocities whole, under 64 MB, identically in two calls."""
    import numpy as np
    import torch

    sys.path.insert(0, ROOT)
    import bench

    for layout in ("split", "block"):
        model = _stand_in_model(2_000_000, layout)
        dirs = [tmp_path / f"{layout}{k}" for k in range(2)]
        for d in dirs:
            bench.dump_outputs(str(d), model, torch.tensor(0.25))
        names = sorted(os.listdir(dirs[0]))
        assert names == sorted([k + ".npy" for k in model.params] + ["loss.npy", "cam_vel.npy"])
        assert sum(os.path.getsize(dirs[0] / f) for f in names) <= 64_000_000
        out = {f[:-4]: np.load(dirs[0] / f) for f in names}
        assert all(np.array_equal(out[f[:-4]], np.load(dirs[1] / f)) for f in names)
        assert out["loss"] == np.float32(0.25) and np.array_equal(out["cam_vel"], np.ones((16, 6), np.float32))
        rows = out["means"][:, 0]
        assert 0 < rows.size < 2_000_000 and np.all(np.diff(rows) > 0)
        for k in model.params:
            assert out[k].dtype == np.float32 and np.array_equal(out[k][:, 0], rows), k
