"""CPU-side checks of the drop-in boundary: the C-ABI library builds for sm_100a, loads, exports
every symbol include/nerf_pl_b200.h declares, validates arguments without touching a GPU, and the
Python mirror keeps the reference's names / signatures / state_dict keys."""
import ctypes
import inspect
import os
import re

import pytest
import torch

import nerf_pl_b200 as nb
from nerf_pl_b200 import _lib
from oracle import nerf_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    _lib.build()
    return _lib.load()


def test_header_symbols_exported(lib):
    hdr = open(os.path.join(ROOT, "include", "nerf_pl_b200.h")).read()
    declared = set(re.findall(r"\b(nerfb200_[a-z_0-9]+)\s*\(", hdr))
    declared -= {"nerfb200_render_args", "nerfb200_backward_args"}
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name
    # the diagnostics (include/nerf_pl_b200_diag.h) are NOT in the product library
    diag = open(os.path.join(ROOT, "include", "nerf_pl_b200_diag.h")).read()
    diag_decl = set(re.findall(r"\b(nerfb200_[a-z_0-9]+)\s*\(", diag))
    assert diag_decl == set(_lib.DIAG_EXPORTS), diag_decl ^ set(_lib.DIAG_EXPORTS)
    if not os.environ.get("NERFB200_LIB"):
        for name in diag_decl:
            assert not hasattr(lib, name), name


def test_abi_basics(lib):
    assert lib.nerfb200_abi_version() == 3
    # layout.h: 30 x 32 KiB + 5 x 16 KiB fp16 slices + fp32 tail, rounded to 1 KiB, + 30 backward slices
    fwd = 30 * 32768 + 5 * 16384 + 4 * (9 * 256 + 256 + 4 + 384 + 4 + 28 * 128)
    assert lib.nerfb200_packed_bytes() == (fwd + 1023) // 1024 * 1024 + 30 * 32768
    assert lib.nerfb200_launch_count() >= 0
    # the Python mirrors of the argument structs have the C sizes (x86-64 / aarch64 LP64 layout)
    assert ctypes.sizeof(_lib.RenderArgs) == 8 * 5 + 4 * 2 + 4 + 4 * 2 + 4 * 2 + 4 + 8 * 14 + 8 + 8 * 4 + 8 + 8
    assert ctypes.sizeof(_lib.BackwardArgs) == 8 * 13


def test_struct_mirrors_match_the_header(tmp_path):
    """sizeof / offsetof of the argument structs as gcc lays out include/nerf_pl_b200.h == the ctypes mirrors."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "nerf_pl_b200.h"\n'
                   'int main(void){printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(nerfb200_render_args), '
                   'sizeof(nerfb200_backward_args), offsetof(nerfb200_render_args, rng_seed), '
                   'offsetof(nerfb200_render_args, rng_in_kernel), offsetof(nerfb200_render_args, train_workspace), '
                   'offsetof(nerfb200_render_args, perturb_rand));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.run(["gcc", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    R = _lib.RenderArgs
    assert got == [ctypes.sizeof(R), ctypes.sizeof(_lib.BackwardArgs), R.rng_seed.offset, R.rng_in_kernel.offset,
                   R.train_workspace.offset, R.perturb_rand.offset]


def test_training_workspace_layout(lib):
    """Workspace size is a pure function of the shape: monotone in n_rays, ~9 KiB per ray-sample."""
    b1 = lib.nerfb200_train_workspace_bytes(1024, 64, 64)
    b2 = lib.nerfb200_train_workspace_bytes(2048, 64, 64)
    assert 0 < b1 < b2
    per_sample = (b2 - b1) / (1024 * 192)
    assert 8000 < per_sample < 11000
    assert lib.nerfb200_train_workspace_bytes(0, 64, 64) == 0
    a = _lib.RenderArgs(n_rays=4, n_samples=64, n_importance=0)
    b = _lib.BackwardArgs(render=ctypes.pointer(a))
    assert lib.nerfb200_render_backward(ctypes.byref(b), None) == -1      # NULL rays / tables


def test_argument_validation_without_gpu(lib):
    a = _lib.RenderArgs(n_rays=4, n_samples=48, n_importance=0)
    assert lib.nerfb200_render_rays(ctypes.byref(a), None) == -2          # unsupported N_samples
    assert b"N_samples" in lib.nerfb200_last_error()
    a = _lib.RenderArgs(n_rays=4, n_samples=64, n_importance=64)
    assert lib.nerfb200_render_rays(ctypes.byref(a), None) == -1          # NULL rays
    a = _lib.RenderArgs(n_rays=0, n_samples=64, n_importance=0)
    assert lib.nerfb200_render_rays(ctypes.byref(a), None) == 0           # empty input is a no-op
    assert lib.nerfb200_searchsorted(None, None, None, 3, 2, 4, 4, 1, None) == -1   # row mismatch
    assert lib.nerfb200_searchsorted(None, None, None, 0, 0, 4, 4, 1, None) == 0    # empty
    assert lib.nerfb200_composite(None, None, None, None, None, 0.0, 0, 4, 48, None, None, None, None, None) == -2
    assert lib.nerfb200_nerf_forward(None, 0, 90, None, 0, None, None) == 0
    assert lib.nerfb200_embed(None, 5, 10, None, None) == -1


def test_python_mirror_matches_reference_interface():
    sig = inspect.signature(nb.render_rays)
    names = list(sig.parameters)[:11]
    assert names == ["models", "embeddings", "rays", "N_samples", "use_disp", "perturb", "noise_std",
                     "N_importance", "chunk", "white_back", "test_time"]      # models/rendering.py:58-69
    d = {k: v.default for k, v in sig.parameters.items()}
    assert (d["N_samples"], d["use_disp"], d["perturb"], d["noise_std"], d["N_importance"], d["chunk"],
            d["white_back"], d["test_time"]) == (64, False, 0, 1, 0, 1024 * 32, False, False)
    m = nb.NeRF()
    assert list(m.state_dict().keys()) == orc.PARAM_KEYS                    # models/nerf.py:69-81
    assert sum(p.numel() for p in m.parameters()) == 595844
    e = nb.Embedding(3, 10)
    assert e.out_channels == 63 and nb.Embedding(3, 4).out_channels == 27
    assert torch.equal(e.freq_bands, 2 ** torch.arange(10.0))


def test_no_cpu_fallback():
    m = nb.NeRF()
    emb = [nb.Embedding(3, 10), nb.Embedding(3, 4)]
    with pytest.raises(RuntimeError):
        nb.render_rays([m, m], emb, torch.zeros(4, 8), 64, False, 0, 0, 64)
    with pytest.raises(RuntimeError):
        m(torch.zeros(2, 90))
    with pytest.raises(RuntimeError):
        emb[0](torch.zeros(2, 3))
    with pytest.raises(RuntimeError):
        nb.searchsorted(torch.zeros(1, 3), torch.zeros(1, 3))


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "nerf_pl_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert "oracle" not in src, fn


def test_nerf_parameters_order_matches_state_dict():
    """The packed-image cache reads the 24 parameters through Module._modules / _parameters
    (hot path of every render_rays call); it must see the state_dict order, for this package's
    NeRF and for a module built the way the reference builds its own (models/nerf.py:58-81)."""
    import torch
    from torch import nn

    from nerf_pl_b200.nerf import NeRF, nerf_parameters

    m = NeRF()
    got = nerf_parameters(m)
    want = [p for _, p in m.named_parameters()]
    assert len(got) == 24 and all(a is b for a, b in zip(got, want))

    class RefLike(nn.Module):            # attribute layout of the reference's NeRF
        def __init__(self):
            super().__init__()
            for i in range(8):
                n_in = 63 if i == 0 else (256 + 63 if i == 4 else 256)
                setattr(self, f"xyz_encoding_{i + 1}", nn.Sequential(nn.Linear(n_in, 256), nn.ReLU(True)))
            self.xyz_encoding_final = nn.Linear(256, 256)
            self.dir_encoding = nn.Sequential(nn.Linear(256 + 27, 128), nn.ReLU(True))
            self.sigma = nn.Linear(256, 1)
            self.rgb = nn.Sequential(nn.Linear(128, 3), nn.Sigmoid())

    r = RefLike()
    got = nerf_parameters(r)
    want = [p for _, p in r.named_parameters()]
    assert len(got) == 24 and all(a is b for a, b in zip(got, want))
    assert [tuple(p.shape) for p in got][:2] == [(256, 63), (256,)]
    del torch


def test_bench_b200_arm_does_not_touch_oracle():
    """Only bench.py's cpu_baseline / --impl reference legs may execute oracle/ (it is the thing
    timed there); the measured arm builds its inputs with bench.py's own generators."""
    import ast

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    tree = ast.parse(open(os.path.join(root, "bench.py")).read())
    fns = {n.name: n for n in tree.body if isinstance(n, ast.FunctionDef)}
    for name in ("run_b200", "synthetic_weights", "blender_rays", "main"):
        src = ast.unparse(fns[name])
        # (run_b200 calls cpu_oracle_throughput(): that IS the cpu_baseline leg)
        assert "import oracle" not in src and "from oracle" not in src and "orc." not in src, name
    top = [n for n in tree.body if isinstance(n, (ast.Import, ast.ImportFrom))]
    assert all("oracle" not in ast.unparse(n) for n in top)


def test_bench_reference_arm_prints_one_json_line():
    """bench.py --impl reference (the CPU arm the driver runs next to the GPU arm): exactly one
    JSON line on stdout with the contract's keys."""
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       cwd=root, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    staged = os.path.exists(os.path.join(root, "baseline", "_ref", "models", "rendering.py"))
    assert d["impl"] == "reference" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == ("reference" if staged else "port")
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_bench_dump_outputs_writes_float_arrays(tmp_path, monkeypatch):
    """bench.py --dump-outputs writes float arrays as .npy and refuses other dtypes or more than its size limit
    before writing anything."""
    import numpy as np

    import bench
    a = {"rgb": np.arange(6, dtype=np.float32).reshape(2, 3), "depth": np.ones(2)}
    bench.dump_outputs(str(tmp_path / "d"), a)
    for k, v in a.items():
        got = np.load(tmp_path / "d" / f"{k}.npy")
        assert got.dtype == v.dtype and np.array_equal(got, v)
    with pytest.raises(TypeError):
        bench.dump_outputs(str(tmp_path / "i"), {"n": np.zeros(2, np.int32)})
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 8)
    with pytest.raises(ValueError):
        bench.dump_outputs(str(tmp_path / "big"), a)
    assert not (tmp_path / "i").exists() and not (tmp_path / "big").exists()


@pytest.mark.gpu
def test_bench_dump_outputs_repeat_exactly(tmp_path):
    """Two bench runs with the same arguments render the same inputs: their dumped last-step outputs are equal."""
    import json
    import subprocess
    import sys

    import numpy as np

    dumps = []
    for run in ("a", "b"):
        d = tmp_path / run
        r = subprocess.run([sys.executable, "bench.py", "--steps", "3", "--warmup", "3", "--no-train",
                            "--dump-outputs", str(d)], cwd=ROOT, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 3
        dumps.append({p.stem: np.load(p) for p in sorted(d.glob("*.npy"))})
    shapes = {"rgb_coarse": (1024, 3), "depth_coarse": (1024,), "opacity_coarse": (1024,),
              "rgb_fine": (1024, 3), "depth_fine": (1024,), "opacity_fine": (1024,)}
    assert {k: v.shape for k, v in dumps[0].items()} == shapes
    for k, v in dumps[0].items():
        assert v.dtype == np.float32 and np.isfinite(v).all(), k
        assert np.array_equal(v, dumps[1][k]), k


def test_integration_md_stub_matches_the_struct():
    """The ctypes stub printed in INTEGRATION.md section 4 is the struct the library takes (names, order, size)."""
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    txt = open(os.path.join(root, "INTEGRATION.md")).read()
    block = txt[txt.index("class RenderArgs(ctypes.Structure):"):txt.index("packed = torch.empty(lib.nerfb200_packed_bytes()")]
    assert re.findall(r'\("(\w+)", ctypes\.c_\w+\)', block) == [f[0] for f in _lib.RenderArgs._fields_]
    ns = {}
    exec("import ctypes\n" + block, ns)
    assert ctypes.sizeof(ns["RenderArgs"]) == ctypes.sizeof(_lib.RenderArgs)
