"""Build and load ``libnerf_pl_b200.so`` (the C-ABI library, ``include/nerf_pl_b200.h``).

The library is compiled in-tree with plain ``nvcc`` (no torch headers) so it builds in seconds,
ships to the GPU box with the repository snapshot and shows up as a loaded in-tree ``.so``.
There is no CPU fallback: if the library is missing or cannot be loaded every operator in this
package raises.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import threading
from ctypes import POINTER, c_char_p, c_float, c_int32, c_int64, c_size_t, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(_HERE, "libnerf_pl_b200.so")
if os.environ.get("NERFB200_LIB"):          # experiment builds (tools/build_variants.py); unset in production
    LIB_PATH = os.path.abspath(os.environ["NERFB200_LIB"])
SOURCES = ["capi.cu"]
HEADERS = ["ptx.cuh", "layout.h", "mlp_engine.cuh", "render_kernel.cuh", "aux_kernels.cuh", "bwd_kernels.cuh",
           "diag_kernels.cuh"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "--shared", "-Xcompiler", "-fPIC",
    "-diag-suppress", "550",
]

# Every symbol include/nerf_pl_b200.h declares (tests check the library exports all of them).
EXPORTS = [
    "nerfb200_abi_version",
    "nerfb200_last_error",
    "nerfb200_packed_bytes",
    "nerfb200_pack_weights",
    "nerfb200_pack_weights_pair",
    "nerfb200_render_rays",
    "nerfb200_render_rays_host",
    "nerfb200_nerf_forward",
    "nerfb200_embed",
    "nerfb200_searchsorted",
    "nerfb200_sample_pdf",
    "nerfb200_composite",
    "nerfb200_query_sigma",
    "nerfb200_mse_psnr",
    "nerfb200_train_workspace_bytes",
    "nerfb200_train_workspace_init",
    "nerfb200_render_backward",
    "nerfb200_train_saturation",
    "nerfb200_adam_step",
    "nerfb200_generate_rays",
    "nerfb200_to_uint8",
    "nerfb200_launch_count",
    "nerfb200_check_status",
    "nerfb200_sm_count",
]
# include/nerf_pl_b200_diag.h: only in -DNERFB200_DIAG builds (tools/build_variants.py)
DIAG_EXPORTS = [
    "nerfb200_debug_gemm",
    "nerfb200_debug_gemm_mn",
    "nerfb200_debug_timeline",
    "nerfb200_debug_mma_bench",
    "nerfb200_debug_mma_contention",
]


class RenderArgs(ctypes.Structure):
    """Mirror of ``nerfb200_render_args`` (include/nerf_pl_b200.h)."""

    _fields_ = [
        ("rays", c_void_p),
        ("n_rays", c_int64),
        ("ray_stride", c_int64),
        ("packed_coarse", c_void_p),
        ("packed_fine", c_void_p),
        ("n_samples", c_int32),
        ("n_importance", c_int32),
        ("use_disp", c_int32),
        ("perturb", c_float),
        ("noise_std", c_float),
        ("white_back", c_int32),
        ("test_time", c_int32),
        ("perturb_rand", c_void_p),
        ("noise_coarse", c_void_p),
        ("u_rand", c_void_p),
        ("noise_fine", c_void_p),
        ("rgb_coarse", c_void_p),
        ("depth_coarse", c_void_p),
        ("opacity_coarse", c_void_p),
        ("rgb_fine", c_void_p),
        ("depth_fine", c_void_p),
        ("opacity_fine", c_void_p),
        ("z_fine", c_void_p),
        ("weights_coarse", c_void_p),
        ("weights_fine", c_void_p),
        ("status", c_void_p),
        ("max_ctas", c_int32),
        ("z_coarse", c_void_p),
        ("train_workspace", c_void_p),
        ("target", c_void_p),
        ("loss_out", c_void_p),
        ("rng_seed", ctypes.c_uint64),
        ("rng_in_kernel", c_int32),
    ]


class BackwardArgs(ctypes.Structure):
    """Mirror of ``nerfb200_backward_args`` (include/nerf_pl_b200.h)."""

    _fields_ = [
        ("render", POINTER(RenderArgs)),
        ("params_coarse", POINTER(c_void_p)),
        ("params_fine", POINTER(c_void_p)),
        ("g_rgb_coarse", c_void_p),
        ("g_depth_coarse", c_void_p),
        ("g_opacity_coarse", c_void_p),
        ("g_rgb_fine", c_void_p),
        ("g_depth_fine", c_void_p),
        ("g_opacity_fine", c_void_p),
        ("target", c_void_p),
        ("loss_grad", c_void_p),
        ("grads_coarse", POINTER(c_void_p)),
        ("grads_fine", POINTER(c_void_p)),
    ]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS]
    deps.append(os.path.join(_HERE, "..", "include", "nerf_pl_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile the CUDA library for sm_100a (cross-compiles without a GPU)."""
    if not force and not needs_build():
        return LIB_PATH
    cmd = [_nvcc(), *NVCC_FLAGS, "-o", LIB_PATH] + [os.path.join(CSRC, s) for s in SOURCES]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + proc.stdout + proc.stderr)
    if verbose:
        print(proc.stderr)
    return LIB_PATH


_lib = None
_lock = threading.Lock()


def _declare(lib: ctypes.CDLL) -> None:
    lib.nerfb200_abi_version.restype = c_int32
    lib.nerfb200_last_error.restype = c_char_p
    lib.nerfb200_packed_bytes.restype = c_size_t
    lib.nerfb200_pack_weights.argtypes = [POINTER(c_void_p), c_void_p, c_void_p]
    lib.nerfb200_pack_weights_pair.argtypes = [POINTER(c_void_p), c_void_p, POINTER(c_void_p), c_void_p, c_void_p]
    lib.nerfb200_render_rays.argtypes = [POINTER(RenderArgs), c_void_p]
    lib.nerfb200_render_rays_host.argtypes = [POINTER(RenderArgs), c_void_p]
    lib.nerfb200_nerf_forward.argtypes = [c_void_p, c_int64, c_int64, c_void_p, c_int32, c_void_p, c_void_p]
    lib.nerfb200_embed.argtypes = [c_void_p, c_int64, c_int32, c_void_p, c_void_p]
    lib.nerfb200_searchsorted.argtypes = [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int32,
                                          c_int32, c_int32, c_void_p]
    lib.nerfb200_sample_pdf.argtypes = [c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32,
                                        c_void_p, c_void_p]
    lib.nerfb200_composite.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float,
                                       c_int32, c_int64, c_int32, c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_void_p]
    lib.nerfb200_query_sigma.argtypes = [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p]
    lib.nerfb200_query_sigma.restype = c_int32
    lib.nerfb200_train_workspace_bytes.argtypes = [c_int64, c_int32, c_int32]
    lib.nerfb200_train_workspace_bytes.restype = c_size_t
    lib.nerfb200_train_workspace_init.argtypes = [c_void_p, c_size_t, c_int64, c_int32, c_int32, c_void_p]
    lib.nerfb200_train_workspace_init.restype = c_int32
    lib.nerfb200_render_backward.argtypes = [POINTER(BackwardArgs), c_void_p]
    lib.nerfb200_render_backward.restype = c_int32
    lib.nerfb200_train_saturation.argtypes = [c_void_p, c_int64, c_int32, c_int32, POINTER(ctypes.c_uint32), c_void_p]
    lib.nerfb200_train_saturation.restype = c_int32
    lib.nerfb200_adam_step.argtypes = [c_int32, POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p),
                                       POINTER(c_int64), c_float, c_float, c_float, c_float, c_float, c_int64, c_void_p]
    lib.nerfb200_adam_step.restype = c_int32
    lib.nerfb200_mse_psnr.argtypes = [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]
    lib.nerfb200_mse_psnr.restype = c_int32
    lib.nerfb200_generate_rays.argtypes = [c_int32, c_int32, c_float, POINTER(c_float), c_float, c_float, c_int32,
                                           c_void_p, c_void_p]
    lib.nerfb200_generate_rays.restype = c_int32
    lib.nerfb200_to_uint8.argtypes = [c_void_p, c_int64, c_void_p, c_void_p]
    lib.nerfb200_to_uint8.restype = c_int32
    if hasattr(lib, "nerfb200_debug_gemm"):        # diagnostics build only
        lib.nerfb200_debug_gemm.argtypes = [c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p]
        lib.nerfb200_debug_gemm.restype = c_int32
        lib.nerfb200_debug_gemm_mn.argtypes = [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p]
        lib.nerfb200_debug_gemm_mn.restype = c_int32
        lib.nerfb200_debug_mma_bench.argtypes = [c_void_p, c_int32, c_int32, c_void_p]
        lib.nerfb200_debug_mma_bench.restype = c_int32
        lib.nerfb200_debug_mma_contention.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p]
        lib.nerfb200_debug_mma_contention.restype = c_int32
        lib.nerfb200_debug_timeline.argtypes = [c_void_p, c_int64]
        lib.nerfb200_debug_timeline.restype = c_int32
    lib.nerfb200_check_status.restype = c_int32
    lib.nerfb200_launch_count.restype = c_int64
    lib.nerfb200_sm_count.restype = c_int32
    for name in ("nerfb200_pack_weights", "nerfb200_pack_weights_pair", "nerfb200_render_rays", "nerfb200_render_rays_host",
                 "nerfb200_nerf_forward", "nerfb200_embed", "nerfb200_searchsorted",
                 "nerfb200_sample_pdf", "nerfb200_composite"):
        getattr(lib, name).restype = c_int32


def load() -> ctypes.CDLL:
    """Load the library (never builds implicitly: build() is the explicit step)."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(
                    f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                    "(nerf_pl_b200 has no CPU fallback)")
            lib = ctypes.CDLL(LIB_PATH)
            _declare(lib)
            if lib.nerfb200_abi_version() != 3:
                raise RuntimeError("libnerf_pl_b200.so ABI version mismatch")
            _lib = lib
    return _lib


class NerfB200Error(RuntimeError):
    pass


def check(rc: int, what: str) -> None:
    """Map the C-ABI return code to the Python exceptions the reference raises
    (asserts / Exception in searchsorted.py:23-45, RuntimeError from AT_ASSERTM)."""
    if rc == 0:
        return
    msg = load().nerfb200_last_error().decode("utf-8", "replace")
    if rc in (-1, -2):
        raise ValueError(f"{what}: {msg}")
    raise NerfB200Error(f"{what}: {msg} (code {rc})")
