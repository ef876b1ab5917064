"""CPU-side checks of the boundary: the C-ABI library loads, exports every symbol the header declares, fails
loudly without a GPU, and the module mirror keeps the reference's surface. No compute calls (no GPU here)."""
import ctypes
import math
import os
import re
import subprocess
import sys

import pytest
import torch

from distributed_sigmoid_loss_b200 import DDPSigmoidLoss, SigLipLoss, SigmoidLoss, _capi, chunk_schedule

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    text = open(os.path.join(ROOT, "include", "siglip_b200.h")).read()
    return sorted(set(re.findall(r"\b(siglip_[a-z_0-9]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    L = _capi.lib()
    declared = _header_symbols()
    assert declared, "no declarations parsed from include/siglip_b200.h"
    for sym in declared:
        assert hasattr(L, sym), f"{sym} declared in include/siglip_b200.h but not exported by {_capi.LIB_PATH}"
    assert set(declared) == set(_capi.EXPORTED_SYMBOLS), set(declared) ^ set(_capi.EXPORTED_SYMBOLS)
    assert "sm_100a" in _capi.version()


def test_library_is_sm100a_native():
    """The shipped binary contains tcgen05 / TMA machine code (SASS mnemonics), not a legacy mma.sync path."""
    import shutil
    import subprocess

    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    sass = subprocess.run(["cuobjdump", "-sass", _capi.LIB_PATH], capture_output=True, text=True).stdout
    assert "UTCHMMA" in sass and "UTMALDG" in sass and "LDTM" in sass and "UTMASTG" in sass
    assert "HMMA.16816" not in sass


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_device_fails_loudly():
    L = _capi.lib()
    assert L.siglip_device_count() == 0
    h = ctypes.c_void_p()
    rc = L.siglip_ctx_create(ctypes.byref(h), 0, 0, 1, 64, 64)
    assert rc == _capi.SIGLIP_ERR_NO_DEVICE
    assert "no CPU fallback" in _capi.last_error()
    mod = DDPSigmoidLoss(4)
    with pytest.raises(RuntimeError, match="no CPU path"):
        mod(torch.randn(4, 8), torch.randn(4, 8))


def test_invalid_arguments_are_rejected_before_touching_the_gpu():
    L = _capi.lib()
    h = ctypes.c_void_p()
    assert L.siglip_ctx_create(ctypes.byref(h), 0, 3, 2, 64, 64) == _capi.SIGLIP_ERR_INVALID   # rank >= world
    assert L.siglip_ctx_create(ctypes.byref(h), 0, 0, 1, 64, 60) == _capi.SIGLIP_ERR_INVALID   # D % 8 != 0
    assert L.siglip_ctx_create(ctypes.byref(h), 0, 0, 64, 64, 64) == _capi.SIGLIP_ERR_INVALID  # world > 32
    assert L.siglip_ctx_handle_bytes() > 3 * 64


def test_module_surface_matches_reference():
    """Same parameters, dtypes, init values and state_dict keys as distributed_sigmoid_loss.py:9-15."""
    mod = DDPSigmoidLoss(gpu_batch_size=8)
    assert SigmoidLoss is DDPSigmoidLoss
    sd = mod.state_dict()
    assert list(sd.keys()) == ["t_prime", "bias"]
    assert mod.t_prime.dtype == torch.float64 and mod.t_prime.dim() == 0
    assert mod.bias.dtype == torch.float32 and mod.bias.dim() == 0
    assert abs(float(mod.t_prime) - math.log(10)) < 1e-15 and float(mod.bias) == -10.0
    assert mod.gpu_batch_size == 8
    assert [n for n, _ in mod.named_parameters()] == ["t_prime", "bias"]
    # the reference's checkpoints load unchanged
    mod.load_state_dict({"t_prime": torch.tensor(1.5, dtype=torch.float64), "bias": torch.tensor(-3.0)})
    assert float(mod.t_prime) == 1.5 and float(mod.bias) == -3.0


def test_batch_mismatch_raises_runtime_error_like_reference():
    mod = DDPSigmoidLoss(gpu_batch_size=8)
    with pytest.raises(RuntimeError, match="must match the size"):
        mod(torch.randn(4, 16), torch.randn(4, 16))
    with pytest.raises(RuntimeError, match="same shape"):
        mod(torch.randn(8, 16), torch.randn(6, 16))


def test_siglip_adapter_signature():
    m = SigLipLoss(cache_labels=False, rank=0, world_size=1, bidir=True, use_horovod=False)
    assert (m.rank, m.world_size, m.bidir) == (0, 1, True)
    with pytest.raises(AssertionError):
        SigLipLoss(use_horovod=True)


@pytest.mark.parametrize("bidir", [False, True])
@pytest.mark.parametrize("world", [1, 2, 3, 4, 5, 8])
def test_chunk_schedule_covers_every_pair_once(world, bidir):
    """Every (image rank, text chunk) pair is scored exactly once; step 0 is the own chunk (positives); at every
    step the W ranks read W distinct owners (a permutation: no NVSwitch hot spot). bidir = the visiting order of the
    reference's bidirectional exchange (rwightman_sigmoid_loss.py:75-107): right, left, right+1, left+1, ..."""
    seen = set()
    for r in range(world):
        sched = chunk_schedule(r, world, bidir)
        assert sched[0] == r and sorted(sched) == list(range(world))
        seen.update((r, c) for c in sched)
    assert len(seen) == world * world
    for k in range(world):
        assert sorted(chunk_schedule(r, world, bidir)[k] for r in range(world)) == list(range(world))
    if bidir and world >= 3:
        assert chunk_schedule(0, world, True)[1:3] == [1, world - 1]


def test_reference_copy_for_the_cpu_arm_is_byte_identical(tmp_path, monkeypatch):
    """tools/fetch_ref.py copies the unmodified reference verbatim under the git-ignored baseline/_ref and writes the
    sha256 of every file into a manifest. The recipe is checked on a stand-in source tree; a copy that build() placed
    in this tree must carry the upstream digests pinned in tests/golden/reference_sha256.json."""
    import hashlib
    import json
    import shutil

    sys.path.insert(0, os.path.join(ROOT, "tools"))
    try:
        import fetch_ref
    finally:
        sys.path.pop(0)
    src, dst = tmp_path / "src", tmp_path / "dst"
    src.mkdir()
    for i, name in enumerate(fetch_ref.FILES):
        (src / name).write_bytes(f"# {name}\n".encode() + bytes(range(256)) * (i + 1))
    monkeypatch.setattr(fetch_ref, "DEST", str(dst))
    assert fetch_ref.fetch(str(src), quiet=True)
    manifest = json.load(open(dst / "MANIFEST.json"))["sha256"]
    assert sorted(manifest) == sorted(fetch_ref.FILES)
    for name, digest in manifest.items():
        a, b = (src / name).read_bytes(), (dst / name).read_bytes()
        assert a == b and hashlib.sha256(b).hexdigest() == digest, name

    pinned = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_sha256.json")))["sha256"]
    assert sorted(pinned) == sorted(fetch_ref.FILES)
    copy = os.path.join(ROOT, "baseline", "_ref")
    if os.path.exists(os.path.join(copy, "MANIFEST.json")):
        assert json.load(open(os.path.join(copy, "MANIFEST.json")))["sha256"] == pinned
        for name, digest in pinned.items():
            assert hashlib.sha256(open(os.path.join(copy, name), "rb").read()).hexdigest() == digest, name

    # the directory stays out of the history (checked against the .gitignore alone: a checkout need not be a clone)
    repo = tmp_path / "repo"
    repo.mkdir()
    shutil.copyfile(os.path.join(ROOT, ".gitignore"), repo / ".gitignore")
    subprocess.run(["git", "init", "-q"], cwd=repo, check=True)
    out = subprocess.run(["git", "check-ignore", "baseline/_ref/distributed_sigmoid_loss.py"], cwd=repo,
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stderr


def test_bench_parity_reference_agrees_with_the_pinned_oracle():
    """bench.py's parity block carries its own fp32 torch restatement of distributed_sigmoid_loss.py:22-47 (the bench
    may use oracle/ only for its CPU arm): it must agree with the oracle that is pinned on the reference's fixtures."""
    import importlib.util

    import numpy as np
    import torch

    from oracle.siglip_oracle import closed_form

    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    W, B, D = 3, 24, 40
    g = torch.Generator().manual_seed(3)
    img_all = torch.nn.functional.normalize(torch.randn(W * B, D, generator=g))
    txt_all = torch.nn.functional.normalize(torch.randn(W * B, D, generator=g))
    tp, bias = math.log(12.0), -7.5
    ref = closed_form(img_all.numpy(), txt_all.numpy(), tp, bias, W)
    contrib = [None] * W
    for r in range(W):
        loss, dimg, cs, dtp, db = bench._fp32_autograd(img_all[r * B:(r + 1) * B],
                                                       [txt_all[c * B:(c + 1) * B] for c in range(W)], tp, bias, r)
        assert abs(loss - ref[r]["loss"]) <= 1e-5 * abs(ref[r]["loss"])
        assert abs(dtp - ref[r]["dt_prime"]) <= 1e-4 * abs(ref[r]["dt_prime"])
        assert abs(db - ref[r]["dbias"]) <= 1e-4 * abs(ref[r]["dbias"])
        assert np.allclose(dimg.numpy(), ref[r]["dimg"], rtol=1e-4, atol=1e-7)
        contrib[r] = cs
    for c in range(W):       # text gradient = sum over the ranks' contributions (the all_reduce in bench.py)
        total = sum(contrib[r][c] for r in range(W))
        assert np.allclose(total.numpy(), ref[c]["dtxt"], rtol=1e-4, atol=1e-7)


def test_module_pads_odd_widths_and_copies_views_without_a_gpu():
    import torch

    from distributed_sigmoid_loss_b200.loss import _aligned, _pad_dim

    x = torch.randn(6, 5, requires_grad=True)
    y = _pad_dim(x)
    assert y.shape == (6, 8) and torch.equal(y[:, :5], x) and float(y[:, 5:].abs().sum()) == 0.0
    y.sum().backward()
    assert x.grad.shape == (6, 5)                       # the gradient comes back sliced
    assert _pad_dim(torch.zeros(3, 16)).shape == (3, 16)
    base = torch.zeros(4, 19, dtype=torch.bfloat16)
    v = base[:, 3:11]
    a = _aligned(v)
    assert a.is_contiguous() and a.data_ptr() % 16 == 0 and torch.equal(a, v)


def test_option_and_status_constants_match_the_header():
    """The ctypes binding repeats the enum values of include/siglip_b200.h: a renumbered or missing option would silently
    set the wrong knob."""
    text = open(os.path.join(ROOT, "include", "siglip_b200.h")).read()
    declared = dict((m.group(1), int(m.group(2))) for m in re.finditer(r"\b(SIGLIP_(?:OPT|ERR)_[A-Z0-9_]+|SIGLIP_OK)\s*=\s*(\d+)", text))
    assert len([k for k in declared if k.startswith("SIGLIP_OPT_")]) >= 20
    for name, value in declared.items():
        assert hasattr(_capi, name), f"{name} is declared in the header but missing from _capi.py"
        assert getattr(_capi, name) == value, (name, getattr(_capi, name), value)
    values = [v for k, v in declared.items() if k.startswith("SIGLIP_OPT_")]
    assert len(values) == len(set(values)), "two options share a number"
