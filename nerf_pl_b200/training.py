"""Training path of ``render_rays`` (reference: train.py:103-117 — ``results = render_rays(...)``,
``loss = MSELoss(results, rgbs)``, ``loss.backward()`` through models/rendering.py + models/nerf.py):
a ``torch.autograd.Function`` around the fused sm_100a kernels.  No torch op, cuBLAS call or
autograd graph is involved in either direction.

forward : ONE fused ``render_rays_kernel`` launch in training mode.  It renders exactly like
          inference and additionally leaves in the training workspace, per sample, what the backward
          needs: encoded input + the 8 hidden activations (fp16, in the tensor core's MN-major
          operand layout), ReLU sign bits, the direction-layer output, raw sigma / rgb, the depths.
          Optionally the MSE loss / PSNR of the batch are reduced in the same launch
          (``render_rays_loss``).
backward: ``nerfb200_render_backward`` (include/nerf_pl_b200.h): compositing backward -> rgb head ->
          tcgen05 dgrad chain -> tcgen05 split-K wgrad -> fixed-order reduction -> unfolding of the
          packed final.dir layer; fills the 48 ``.grad`` tensors.
The sampling of the fine depths carries no gradient (models/rendering.py:225-227 ``.detach()``).
"""
from __future__ import annotations

import ctypes
import weakref
from typing import Dict, List, Optional

import torch

from . import _lib
from .nerf import _stream_ptr, nerf_parameters, packed_weights, packed_weights_pair


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


class TrainWorkspace:
    """Device workspace of one (device, n_rays, N_samples, N_importance) shape, reused across steps.
    ``busy`` is set between a forward and its backward so that a second forward (gradient
    accumulation over several batches) gets its own buffer.  It is cleared by the backward, or when
    the forward's autograd graph is freed without one (a skipped step, a forward under grad for logging)."""

    _pool: Dict[tuple, List["TrainWorkspace"]] = {}

    def __init__(self, dev: torch.device, n: int, S_c: int, K: int) -> None:
        lib = _lib.load()
        self.bytes = int(lib.nerfb200_train_workspace_bytes(n, S_c, K))
        if self.bytes == 0:
            raise ValueError("invalid training shape")
        raw = torch.empty(self.bytes + 1024, dtype=torch.uint8, device=dev)
        off = (-raw.data_ptr()) % 1024
        self.raw = raw
        self.buf = raw[off:off + self.bytes]
        self.busy = False
        self.shape = (n, S_c, K)
        self.device = dev
        with torch.cuda.device(dev):
            _lib.check(lib.nerfb200_train_workspace_init(self.buf.data_ptr(), self.bytes, n, S_c, K, _stream_ptr()),
                       "nerfb200_train_workspace_init")

    @classmethod
    def acquire(cls, dev: torch.device, n: int, S_c: int, K: int) -> "TrainWorkspace":
        key = (dev.index, n, S_c, K)
        free = cls._pool.setdefault(key, [])
        for ws in free:
            if not ws.busy:
                ws.busy = True
                return ws
        ws = cls(dev, n, S_c, K)
        ws.busy = True
        free.append(ws)
        return ws

    def release(self) -> None:
        self.busy = False

    def saturated(self):
        """(coarse, fine) count of fp16 gradient elements the last backward on this workspace clipped at
        the fp16 limit or stored as NaN (``nerfb200_train_saturation``).  Synchronises the current stream."""
        out = (ctypes.c_uint32 * 2)()
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().nerfb200_train_saturation(self.buf.data_ptr(), *self.shape, out, _stream_ptr()),
                       "nerfb200_train_saturation")
        return int(out[0]), int(out[1])

    @classmethod
    def clear(cls) -> None:
        cls._pool.clear()


def _render_args(cfg, rays, pr, nc, ur, nf, out, blob_c, blob_f, ws, target, loss_out) -> _lib.RenderArgs:
    K = cfg["N_importance"]
    return _lib.RenderArgs(
        rays=rays.data_ptr(), n_rays=rays.shape[0], ray_stride=rays.stride(0),
        packed_coarse=blob_c.data_ptr(), packed_fine=_ptr(blob_f),
        n_samples=cfg["N_samples"], n_importance=K, use_disp=int(cfg["use_disp"]), perturb=cfg["perturb"],
        noise_std=cfg["noise_std"], white_back=int(cfg["white_back"]), test_time=0,
        perturb_rand=_ptr(pr), noise_coarse=_ptr(nc), u_rand=_ptr(ur), noise_fine=_ptr(nf),
        rgb_coarse=out[0].data_ptr(), depth_coarse=out[1].data_ptr(), opacity_coarse=out[2].data_ptr(),
        rgb_fine=_ptr(out[3]) if K > 0 else None, depth_fine=_ptr(out[4]) if K > 0 else None,
        opacity_fine=_ptr(out[5]) if K > 0 else None,
        z_fine=None, weights_coarse=None, weights_fine=None, status=None, max_ctas=0, z_coarse=None,
        train_workspace=ws.buf.data_ptr(), target=_ptr(target), loss_out=_ptr(loss_out),
        rng_seed=cfg.get("rng_seed") or 0, rng_in_kernel=int(cfg.get("rng_seed") is not None))


class FusedRenderFunction(torch.autograd.Function):
    """rays + pre-drawn randoms [+ target] + 48 parameter tensors -> the six result tensors [+ loss4]."""

    @staticmethod
    def forward(ctx, cfg: Dict, rays, pr, nc, ur, nf, target, *params):
        models = cfg["models"]
        S_c, K = cfg["N_samples"], cfg["N_importance"]
        n = rays.shape[0]
        dev = rays.device
        f32 = dict(dtype=torch.float32, device=dev)
        out = [torch.empty(n, 3, **f32), torch.empty(n, **f32), torch.empty(n, **f32)]
        if K > 0:
            out += [torch.empty(n, 3, **f32), torch.empty(n, **f32), torch.empty(n, **f32)]
        loss_out = torch.empty(4, **f32) if target is not None else None
        lib = _lib.load()
        if K > 0:
            blob_c, blob_f = packed_weights_pair(models[0], models[1])      # one launch for both images
        else:
            blob_c, blob_f = packed_weights(models[0]), None
        ws = TrainWorkspace.acquire(dev, n, S_c, K)
        args = _render_args(cfg, rays, pr, nc, ur, nf, out, blob_c, blob_f, ws, target, loss_out)
        with torch.cuda.device(dev):
            _lib.check(lib.nerfb200_render_rays(ctypes.byref(args), _stream_ptr()), "nerfb200_render_rays")
        ctx.cfg = cfg
        # detached views of the outputs: the outputs themselves would close a reference cycle through ctx
        ctx.keep = (rays, pr, nc, ur, nf, target, [o.detach() for o in out], blob_c, blob_f, ws)
        ctx.release_ws = weakref.finalize(ctx, ws.release)      # also runs if the graph dies without a backward
        ctx.n_params = len(params)
        ctx.save_for_backward(*params)
        ctx.set_materialize_grads(False)
        res = tuple(out)
        if loss_out is not None:
            res = res + (loss_out,)
        return res

    @staticmethod
    def backward(ctx, *gouts):
        cfg = ctx.cfg
        params = list(ctx.saved_tensors)
        rays, pr, nc, ur, nf, target, out, blob_c, blob_f, ws = ctx.keep
        K = cfg["N_importance"]
        dev = rays.device
        lib = _lib.load()
        g = [None if t is None else t.detach().to(torch.float32).contiguous() for t in gouts]
        g6 = g[:6] + [None] * (6 - min(len(g), 6))
        if K == 0:
            g6 = g[:3] + [None] * 3
        n_out = 6 if K > 0 else 3
        loss_grad = None
        use_target = None
        if target is not None:
            g4 = g[n_out]
            if g4 is not None:
                # d(loss_out)/d(rgb): element 2 = MSELoss (elements 0 / 1 = its coarse / fine terms: the same
                # seed restricted to one pass is not provided); take the gradient of the total loss
                loss_grad = g4          # the kernel reads element 2 (address passed below)
                use_target = target
        # one allocation for all gradients (the kernels write every element), views per parameter
        sizes, shapes = _param_sizes(params)
        flat = torch.empty(sum(sizes), dtype=torch.float32, device=dev)
        grads = [t.view(shp) for t, shp in zip(flat.split(sizes), shapes)]
        base, offs = flat.data_ptr(), _offsets(sizes)
        pc = (ctypes.c_void_p * 24)(*[p.data_ptr() for p in params[:24]])
        gc = (ctypes.c_void_p * 24)(*[base + 4 * o for o in offs[:24]])
        pf = gf = None
        if K > 0:
            pf = (ctypes.c_void_p * 24)(*[p.data_ptr() for p in params[24:48]])
            gf = (ctypes.c_void_p * 24)(*[base + 4 * o for o in offs[24:48]])
        rargs = _render_args(cfg, rays, pr, nc, ur, nf, out, blob_c, blob_f, ws, None, None)
        bargs = _lib.BackwardArgs(
            render=ctypes.pointer(rargs), params_coarse=pc, params_fine=pf,
            g_rgb_coarse=_ptr(g6[0]), g_depth_coarse=_ptr(g6[1]), g_opacity_coarse=_ptr(g6[2]),
            g_rgb_fine=_ptr(g6[3]), g_depth_fine=_ptr(g6[4]), g_opacity_fine=_ptr(g6[5]),
            target=_ptr(use_target), loss_grad=None if loss_grad is None else loss_grad.data_ptr() + 8,
            grads_coarse=gc, grads_fine=gf)
        with torch.cuda.device(dev):
            _lib.check(lib.nerfb200_render_backward(ctypes.byref(bargs), _stream_ptr()), "nerfb200_render_backward")
        ctx.release_ws()
        ctx.keep = None
        if K == 0:
            grads = grads[:24] + [None] * (ctx.n_params - 24)
        return (None, None, None, None, None, None, None, *grads)


_SIZE_CACHE: Dict[int, tuple] = {}


def _param_sizes(params):
    key = len(params)
    hit = _SIZE_CACHE.get(key)
    if hit is None:
        hit = ([p.numel() for p in params], [tuple(p.shape) for p in params])
        _SIZE_CACHE[key] = hit
    return hit


def _offsets(sizes):
    out, o = [], 0
    for n in sizes:
        out.append(o)
        o += n
    return out


def _params_of(models, N_importance) -> List[torch.Tensor]:
    params = nerf_parameters(models[0])
    if N_importance > 0:
        params = params + nerf_parameters(models[1])
    return params          # shapes / contiguity are validated by packed_weights()


def render_rays_train(models, rays, N_samples, use_disp, perturb, noise_std, N_importance, white_back,
                      pr, nc, ur, nf, target: Optional[torch.Tensor] = None,
                      rng_seed: Optional[int] = None) -> Dict[str, torch.Tensor]:
    """Differentiable render_rays (test_time=False) through FusedRenderFunction.  With ``target``
    (n,3) the result also carries ``loss`` (losses.py:9-14 MSELoss of the batch), ``psnr``
    (metrics.py:4-13, of the finest pass), ``mse_coarse`` and ``mse_fine`` computed by the same
    launch; ``loss.backward()`` then seeds the backward inside the kernels."""
    cfg = dict(models=list(models), N_samples=int(N_samples), N_importance=int(N_importance),
               use_disp=bool(use_disp), perturb=float(perturb), noise_std=float(noise_std),
               white_back=bool(white_back), rng_seed=rng_seed)
    params = _params_of(models, N_importance)
    if target is not None:
        target = target.detach().to(torch.float32).contiguous()
        if target.shape != (rays.shape[0], 3):
            raise ValueError("target must be (N_rays, 3)")
    outs = FusedRenderFunction.apply(cfg, rays, pr, nc, ur, nf, target, *params)
    res = {"rgb_coarse": outs[0], "depth_coarse": outs[1], "opacity_coarse": outs[2]}
    k = 3
    if N_importance > 0:
        res.update(rgb_fine=outs[3], depth_fine=outs[4], opacity_fine=outs[5])
        k = 6
    if target is not None:
        l4 = outs[k]
        res.update(loss=l4[2], psnr=l4[3].detach(), mse_coarse=l4[0].detach(), mse_fine=l4[1].detach())
    return res
