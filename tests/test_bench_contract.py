"""bench.py's output contract (one JSON line, the keys the driver reads). The reference arm runs anywhere (CPU);
this repo's arm needs a B200."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e"}


def _run(args, timeout=900):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                         timeout=timeout, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout
    return json.loads(lines[0])


def test_reference_arm_line():
    """`--impl reference` runs the UNMODIFIED reference module from baseline/_ref (tools/fetch_ref.py) when it is there
    (it is in the build container, and it ships to the GPU box), the oracle port otherwise; a timed step is the full
    per-rank chunk, so steps x ms_per_step is the time the arm really spent."""
    have_ref = os.path.exists(os.path.join(ROOT, "baseline", "_ref", "distributed_sigmoid_loss.py"))
    d = _run(["--impl", "reference", "--gpus", "1", "--steps", "2", "--warmup", "1", "--batch", "256", "--dim", "64"])
    assert d["impl"] == "reference" and BASE_KEYS <= set(d)
    assert d["metric"] == "image-text pairs/sec" and d["unit"] == "pairs/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["gpu_launches"] == 0 and d["steps"] == 2 and d["warmup"] == 1
    cb = d["cpu_baseline"]
    assert cb["kind"] == ("reference" if have_ref else "port")
    assert cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]
    # N = 1: the measured step IS the whole job
    assert abs(d["value"] - 256 / (d["ms_per_step"] * 1e-3)) <= 1e-6 * d["value"]
    # loss of the reference on the bench inputs: the product arm must print the same number (bench.py `loss`)
    assert 5.0 < d["loss"] < 20.0


def test_reference_arm_extrapolates_at_n_gt_1():
    d = _run(["--impl", "reference", "--gpus", "4", "--steps", "1", "--warmup", "0", "--batch", "128", "--dim", "64"])
    # one timed step is still ONE (B x B) chunk; the whole job is W ranks x W chunks of it on this host
    assert abs(d["extrapolated_job_step_ms"] - 16 * d["ms_per_step"]) <= 1e-9 * d["ms_per_step"] * 16
    assert abs(d["value"] - 4 * 128 / (d["extrapolated_job_step_ms"] * 1e-3)) <= 1e-6 * d["value"]
    assert "extrapolated" in d["cpu_baseline"]["sample"]


def _bench_module():
    import importlib.util

    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True,
                         text=True, timeout=60, cwd=ROOT)
    assert out.returncode == 2 and "--steps must be at least 1" in out.stderr


@pytest.mark.parametrize("B,D", [(48, 40), (16384, 1024)])
def test_dump_outputs_files(tmp_path, B, D):
    """What --dump-outputs writes for one step's outputs: float32 / float64 .npy files, at most 64 MB in all; a gradient
    too large for that is cut to the same seeded rows in every run."""
    import numpy as np
    import torch

    bench = _bench_module()
    g = torch.Generator().manual_seed(5)
    outputs = (torch.tensor(9.25), torch.randn(B, D, generator=g).to(torch.bfloat16),
               torch.randn(B, D, generator=g).to(torch.bfloat16), torch.tensor(-0.5, dtype=torch.float64),
               torch.tensor(0.75))
    bench.dump_outputs(str(tmp_path / "a"), outputs)
    bench.dump_outputs(str(tmp_path / "b"), outputs)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(n + ".npy" for n in bench.DUMP_NAMES + ("grad_rows",))
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in names) <= 64e6
    z = {f[:-4]: np.load(tmp_path / "a" / f) for f in names}
    assert all(v.dtype in (np.float32, np.float64) for v in z.values())
    assert z["dt_prime"].dtype == np.float64 and z["loss"].dtype == np.float32
    assert float(z["loss"]) == 9.25 and float(z["dt_prime"]) == -0.5 and float(z["dbias"]) == 0.75
    rows = z["grad_rows"].astype(np.int64)
    assert len(rows) == min(B, bench.DUMP_GRAD_ELEMENTS // D) and np.all(np.diff(rows) > 0)
    for i, name in ((1, "dimg"), (2, "dtxt")):
        assert np.array_equal(z[name], outputs[i].float().numpy()[rows])
    for f in names:
        assert np.array_equal(np.load(tmp_path / "b" / f), z[f[:-4]])


@pytest.mark.gpu
def test_product_arm_line(tmp_path):
    d = _run(["--gpus", "1", "--steps", "3", "--warmup", "3", "--batch", "2048", "--dim", "256", "--sustain-ms", "50",
              "--cpu-steps", "1", "--dump-outputs", str(tmp_path)])
    assert "impl" not in d and BASE_KEYS | {"gpu_launches", "clocks", "roofline", "cpu_baseline", "burst", "parity",
                                            "per_rank"} <= set(d)
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["warmup"] >= 3 and d["dtype"] == "bf16"
    assert d["gpu_launches"] == 2 * 3          # one loss kernel + one gradient kernel per step
    r = d["roofline"]
    assert r["bound"] == "tensor" and r["unit"] == "TFLOP/s" and 0 < r["frac"] < 1.2 and r["launches_timed"] == 3
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] == 2 * 2048 * 256 * 2 and e["d2h_bytes_per_step"] == 12 and e["value"] > 0
    assert e["first_steps_ms_per_step"] > 0 and "sustained" in e["api"]   # the headline e2e figure is the sustained one
    g = e["with_grads"]
    assert g["d2h_bytes_per_step"] == 2 * 2048 * 256 * 2 + 12 and g["value"] > 0 and g["loss"] == e["loss"]
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["value"] > 0
    assert d["clocks"]["samples"] >= 1
    par = d["parity"]
    assert par["pass"] is True and par["shape"] == [2048, 768]
    assert all(v <= 1e-3 for v in par["fused_fp32"].values())
    # --dump-outputs: the last timed step's module outputs (bf16 gradients), against fp32 autograd on the bench inputs
    import numpy as np

    bench = _bench_module()
    z = {n: np.load(tmp_path / (n + ".npy")) for n in bench.DUMP_NAMES + ("grad_rows",)}
    assert float(z["loss"]) == d["loss"]
    assert z["dimg"].shape == z["dtxt"].shape == (2048, 256) and np.array_equal(z["grad_rows"], np.arange(2048))
    img, txt = bench.synth(0, 2048, 256)
    loss, dimg, dtxt, dtp, db = bench._fp32_autograd(img, [txt], np.log(10.0), -10.0, 0)
    dtxt = dtxt[0]
    assert abs(float(z["loss"]) - loss) <= 1e-3 * abs(loss)
    assert abs(float(z["dt_prime"]) - dtp) <= 1e-3 * abs(dtp) and abs(float(z["dbias"]) - db) <= 1e-3 * abs(db)
    for got, ref in ((z["dimg"], dimg), (z["dtxt"], dtxt)):
        assert np.linalg.norm(got - ref.numpy()) <= 4e-3 * np.linalg.norm(ref.numpy())
