"""CPU: the C-ABI library loads without a GPU and exports every symbol include/rbunet.h declares; the product package
imports nothing from oracle/ and has no CPU fallback."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "eusipco-2026-robust-unet_b200")


def test_library_exports_every_declared_symbol():
    from rbunet import _lib
    sigs = _lib.parse_header()
    assert len(sigs) >= 35
    handle = ctypes.CDLL(_lib.LIB_PATH)
    for name in sigs:
        assert hasattr(handle, name), f"{name} declared in rbunet.h but not exported"
    assert _lib.lib().rbu_version() >= 100
    assert _lib.lib().rbu_last_error() is not None


def test_header_prototypes_parse_to_ctypes():
    from rbunet import _lib
    sigs = _lib.parse_header()
    res, args = sigs["rbu_conv_gemm"]
    assert res is ctypes.c_int and args == [ctypes.c_void_p, ctypes.c_void_p]
    res, args = sigs["rbu_loss_workspace_bytes"]
    assert res is ctypes.c_size_t and args == [ctypes.c_int, ctypes.c_int64]
    assert sigs["rbu_launch_count"][0] is ctypes.c_ulonglong


def test_product_never_imports_the_oracle():
    for fn in os.listdir(PKG):
        if fn.endswith(".py"):
            src = open(os.path.join(PKG, fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle", src, flags=re.M), fn


def test_no_cpu_fallback():
    import torch
    import rbunet
    model = rbunet.RobustUNet(3, 1, 16)
    with pytest.raises(RuntimeError):
        model(torch.zeros((1, 3, 32, 32)))
    with pytest.raises(RuntimeError):
        rbunet.RobustBCEDiceLoss()(torch.rand((1, 1, 4, 4)), torch.rand((1, 1, 4, 4)))
    with pytest.raises(RuntimeError):
        rbunet.confusion_counts(torch.rand((1, 4)), torch.rand((1, 4)))


def test_state_dict_schema_and_init_match_the_reference_schema(golden_dir):
    import numpy as np
    import torch
    import rbunet
    from oracle import robust_unet_ref as R
    for nc, golden in ((3, "model_c3_b64_64x64.npz"), (4, "model_c4_b64_64x96.npz")):
        m = rbunet.RobustUNet(nc, 1, 64)
        sd = m.state_dict()
        shapes = R.robust_unet_shapes(nc, 1, 64)
        assert list(sd.keys()) == list(shapes.keys()) and len(sd) == 290
        for k, v in sd.items():
            assert tuple(v.shape) == tuple(shapes[k]), k
        # the reference's parameter and running-statistics names in its registration order (recorded from
        # Main_Final.RobustUNet by oracle/make_golden.py): the same order draws the same initial weights under one seed
        g = np.load(os.path.join(golden_dir, golden))
        assert [n for n, _ in m.named_parameters()] == [str(n) for n in g["param_names"]]
        assert [n for n in sd if n.endswith(("running_mean", "running_var"))] == [str(n) for n in g["buffer_names"]]
    assert sum(p.numel() for p in rbunet.RobustUNet(3).parameters()) == 40872223      # SURVEY.md §2


def test_bench_input_generator_matches_the_oracle_generator():
    """bench.py's product arm uses tools/synthetic.py (no oracle import); it must produce the oracle's tensors."""
    import torch
    from oracle import robust_unet_ref as R
    from tools.synthetic import synthetic_batch
    for (b, c, h, w, seed) in ((2, 3, 32, 48, 123), (1, 4, 16, 16, 7)):
        x, y = synthetic_batch(b, c, h, w, seed=seed)
        xo, yo = R.synthetic_inputs(b, c, h, w, seed=seed, blobby=True)
        assert torch.equal(x, xo) and torch.equal(y, yo)


def test_bench_product_arm_does_not_import_the_oracle():
    src = open(os.path.join(ROOT, "bench.py")).read()
    own = src[src.index("class Env"):src.index("def load_reference_module")]
    assert "oracle" not in own


def test_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours) on a tiny sample: one JSON line with the
    contract's keys, `impl: reference`, a cpu_baseline describing the run and an e2e record with zero copy bytes.  It
    runs the staged reference (`baseline/_ref`, kind "reference") when build() has staged it, else the oracle port."""
    import json
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--size", "32"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "train_images_per_sec" and d["unit"] == "img/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0
