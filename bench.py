"""bench.py — ray-samples/s of the render_rays hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    torchrun --nproc-per-node N ... bench.py --gpus N ...        (one rank per GPU, NCCL)

Workload (BASELINE.json configs[1] at N=1; configs[4]'s training shape at N>1 = the same 1024 rays
per GPU): Blender-lego-shaped 400x400 pinhole rays, N_samples=64, N_importance=64, batch_size=1024
rays per GPU per step, perturb=1, noise_std=0, white_back, coarse rgb computed (test_time=False)
= 1024 x (64 + 128) = 196,608 MLP evaluations per GPU per step.  Synthetic rays / random-init
(pseudo-trained) weights: no dataset or checkpoint on the box.

One JSON line on stdout (rank 0):
  value      device-timed whole-job ray-samples/s of the render_rays forward, batch resident in HBM.
             A "step" = one render_rays pass over one batch (its stratified-sampling random numbers are
             Philox draws inside the kernel: randoms="kernel"); for
             N>1 every step ends with ONE NCCL all-gather of the rendered batch (north_star).  The K
             timed steps are captured in one CUDA graph (no host in the timed region) and bracketed
             by two events; every step reads a different copy of the packed weights and a different
             ray batch, 200+ MB in rotation (> the 126 MB L2), so no step finds its inputs in L2.
  e2e        the same metric through the public Python API with pinned HOST buffers: H2D of the
             rays, render_rays, D2H of all six result tensors, host sync every step.
  train      config 2 as BASELINE.json labels it ("training"): forward with the fused loss +
             hand-written sm_100a backward + Adam, ms per 1024-ray step.
  roofline   the fused forward kernel against the measured dense tensor peak (algorithmic and
             executed FLOPs, burst and sustained), cpu_baseline = the reference's own PyTorch path
             timed on the host cores, parity = the timed batch's first rays checked against it.
  image_800  configs[4] inference: one 800x800 view, contiguous ray shards + one all-gather.
`--impl reference` times the unmodified reference (baseline/_ref, staged by tools/stage_reference.py)
on the host cores; if it is absent, the numpy oracle port (oracle/) — `cpu_baseline.kind` says which.

`--dump-outputs DIR` writes the six float32 result tensors of the last timed step (at N>1 also the
all-gathered batch, `all_gather`) to DIR/<name>.npy.  The inputs are seeded, so two runs with the same
arguments render the same rays with the same random numbers, and two builds can be compared output for output.
The benchmark writes nothing into the repository tree.
"""
import argparse
import json
import os
import sys
import threading
import time
import types

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_SAMPLES, N_IMPORTANCE = 64, 64
BATCH = 1024
SAMPLES_PER_RAY = N_SAMPLES + (N_SAMPLES + N_IMPORTANCE)          # 192 (SURVEY.md section 8d)
FLOP_PER_SAMPLE = 2 * 593408                                     # algorithmic (BASELINE.md section 3)
FLOP_PER_RAY_TRAIN = 192 * FLOP_PER_SAMPLE                        # test_time=False
IMG_W = IMG_H = 400
CAMERA_ANGLE_X = 0.6911112070083618                              # lego transforms_*.json
N_ROT = 96                                                       # weight / ray-batch copies in rotation


def executed_flop_per_sample():
    """MACs the kernel's tensor core actually executes per MLP evaluation (csrc/layout.h): K padded to
    64 / 320, xyz_encoding_final folded into dir_encoding (256x256 + 256x128 -> 256x128), the
    direction part (27x128) and both heads (256 + 384) evaluated on the CUDA cores."""
    macs = 64 * 256 + 3 * 256 * 256 + 320 * 256 + 3 * 256 * 256 + 256 * 128
    return 2 * macs


def blender_rays(n, seed, W=IMG_W, H=IMG_H, pixels=None):
    """n rays of a Blender-style pinhole camera on a radius-4 sphere looking at the origin: unit
    directions, near=2, far=6 (reference datasets/ray_utils.py:5-43, blender.py:28-35).
    Random pixels, or all H*W pixels in row-major order with pixels='all'."""
    rs = np.random.RandomState(seed)
    focal = 0.5 * W / np.tan(0.5 * CAMERA_ANGLE_X)
    th, ph = rs.uniform(0, 2 * np.pi), rs.uniform(np.pi / 6, np.pi / 3)
    cam = 4.0 * np.array([np.cos(th) * np.sin(ph), np.sin(th) * np.sin(ph), np.cos(ph)])
    fwd = -cam / np.linalg.norm(cam)
    right = np.cross(fwd, np.array([0.0, 0.0, 1.0])); right /= np.linalg.norm(right)
    up = np.cross(right, fwd)
    if pixels == "all":
        py, px = np.divmod(np.arange(H * W), W)
        n = H * W
    else:
        px = rs.randint(0, W, n); py = rs.randint(0, H, n)
    dc = np.stack([(px - W / 2) / focal, -(py - H / 2) / focal, -np.ones(n)], -1)
    d = dc[:, :1] * right + dc[:, 1:2] * up - dc[:, 2:3] * fwd
    d /= np.linalg.norm(d, axis=-1, keepdims=True)
    o = np.broadcast_to(cam, (n, 3))
    return np.concatenate([o, d, np.full((n, 1), 2.0), np.full((n, 1), 6.0)], -1).astype(np.float32)


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region, in-process through NVML
    (nvidia-smi's own start-up is longer than a short timed region), every ~2 ms."""

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.stop_flag, self.thread, self.err = gpu_index, [], False, None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.gpu
            if vis:
                try:
                    idx = int(vis.split(",")[self.gpu])
                except Exception:
                    idx = self.gpu
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nv = pynvml
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:          # noqa: BLE001
            self.err = repr(e)
            return
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def _run(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((sm, rs))
            except Exception as e:      # noqa: BLE001
                self.err = repr(e)
                return
            time.sleep(0.002)

    def stop(self):
        self.stop_flag = True
        if self.thread is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + str(self.err)]}
        self.thread.join(timeout=1)
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        reasons = sorted(k for k, bit in names.items() if any(r[1] & bit for r in self.rows))
        sm = [r[0] for r in self.rows]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(self.max_sm),
                "reasons": reasons, "samples": len(sm)}


_NERF_LAYERS = ([("xyz_encoding_1.0", 256, 63)] + [(f"xyz_encoding_{i}.0", 256, 256) for i in (2, 3, 4)]
                + [("xyz_encoding_5.0", 256, 319)] + [(f"xyz_encoding_{i}.0", 256, 256) for i in (6, 7, 8)]
                + [("xyz_encoding_final", 256, 256), ("dir_encoding.0", 128, 283), ("sigma", 1, 256), ("rgb.0", 3, 128)])


def synthetic_weights(seed):
    """Random-init NeRF state_dict (numpy): nn.Linear's default U(-1/sqrt(fan_in), 1/sqrt(fan_in)) for the
    reference architecture (models/nerf.py:58-81), with the sigma / rgb heads scaled so that
    opacities and colours are not degenerate (there are no checkpoints to load).  bench.py's own
    generator: the b200 arm does not touch oracle/."""
    rs = np.random.RandomState(seed)
    w = {}
    for name, out_f, in_f in _NERF_LAYERS:
        bound = 1.0 / np.sqrt(in_f)
        w[name + ".weight"] = rs.uniform(-bound, bound, size=(out_f, in_f)).astype(np.float32)
        w[name + ".bias"] = rs.uniform(-bound, bound, size=(out_f,)).astype(np.float32)
    w["sigma.weight"] = (w["sigma.weight"] * np.float32(30.0)).astype(np.float32)
    w["sigma.bias"] = (w["sigma.bias"] + np.float32(0.5)).astype(np.float32)
    w["rgb.0.weight"] = (w["rgb.0.weight"] * np.float32(8.0)).astype(np.float32)
    return w


def ncu_profile():
    """Numbers of the committed ncu --set full capture of the bench-shaped launch
    (profiles/*_ncu_traffic.json, written by tools/summarize_ncu.py): DRAM bytes per launch and the
    tensor-pipe active percentage; (None, None, None) if absent."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_ncu_traffic.json")))
    if not files:
        return None, None, None
    try:
        j = json.load(open(files[-1]))
        return float(j["traffic_bytes_per_launch"]), j.get("tensor_pipe_active_pct"), os.path.basename(files[-1])
    except Exception:
        return None, None, None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return (float(j["bf16_tflops"]), float(j.get("bf16_tflops_sustained", j["bf16_tflops"])),
                "measured (MEASURED_PEAKS.json: cuBLAS bf16 8192^3, burst / 4 s sustained)")
    return 1590.0, 1400.0, "fallback (B200_PROFILING.md: 1.59 PFLOP/s burst, ~1.4 sustained)"


# ----------------------------------------------------------------------------- the reference on the host
_REF = None


def import_reference():
    """The unmodified reference modules staged under baseline/_ref (tools/stage_reference.py), or None."""
    global _REF
    if _REF is not None:
        return _REF or None
    path = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.exists(os.path.join(path, "models", "rendering.py")):
        _REF = False
        return None
    import torch
    shim = types.ModuleType("torchsearchsorted")       # SURVEY.md section 8c: bit-identical on the reference's test grid
    shim.searchsorted = lambda a, v, out=None, side="left": torch.searchsorted(
        a.contiguous(), v.contiguous(), right=(side == "right"))
    sys.modules["torchsearchsorted"] = shim
    sys.path.insert(0, path)
    try:
        from models.nerf import Embedding, NeRF
        from models.rendering import render_rays
        from losses import MSELoss
    except Exception as e:      # noqa: BLE001
        print("reference import failed:", repr(e), file=sys.stderr)
        _REF = False
        return None
    _REF = {"Embedding": Embedding, "NeRF": NeRF, "render_rays": render_rays, "MSELoss": MSELoss}
    return _REF


class HostReference:
    """The CPU arm: the reference's PyTorch path (kind 'reference') or the numpy oracle (kind 'port')."""

    def __init__(self):
        self.ref = import_reference()
        self.kind = "reference" if self.ref else "port"
        self.ws = [synthetic_weights(11), synthetic_weights(12)]
        self.threads = None
        if self.ref:
            import torch
            self.torch = torch
            self.models = []
            for w in self.ws:
                m = self.ref["NeRF"]()
                m.load_state_dict({k: torch.from_numpy(v) for k, v in w.items()})
                self.models.append(m)
            self.emb = [self.ref["Embedding"](3, 10), self.ref["Embedding"](3, 4)]

    def render(self, rays, randoms=None, seed=0):
        """render_rays(perturb=1, noise_std=0, white_back, test_time=False) -> dict of numpy arrays.
        With `randoms` (perturb_rand, u_rand) the draws are replayed exactly (oracle: passed in; torch:
        the global generator is seeded so that rand() returns them — models/rendering.py:203, :39)."""
        if self.ref:
            torch = self.torch
            if randoms is not None:
                torch.manual_seed(seed)
            with torch.no_grad():
                out = self.ref["render_rays"](self.models, self.emb, torch.from_numpy(rays), N_SAMPLES, False, 1.0, 0.0,
                                              N_IMPORTANCE, 1024 * 32, True, test_time=False)
            return {k: v.numpy() for k, v in out.items()}
        from oracle import nerf_oracle as orc
        return orc.render_rays(self.ws, rays, N_SAMPLES, False, 1.0, 0.0, N_IMPORTANCE, True, False, randoms)

    def replay_randoms(self, n, seed):
        """The two uniform draws the reference makes for an n-ray batch after torch.manual_seed(seed)
        (perturb_rand (n,64) at :203, then — noise_std = 0 still draws randn (n,64) at :152 — u (n,64) at :39)."""
        if self.ref:
            torch = self.torch
            torch.manual_seed(seed)
            pr = torch.rand(n, N_SAMPLES)
            torch.randn(n, N_SAMPLES)
            ur = torch.rand(n, N_IMPORTANCE)
            return {"perturb_rand": pr.numpy(), "u_rand": ur.numpy()}
        rs = np.random.RandomState(seed)
        return {"perturb_rand": rs.rand(n, N_SAMPLES).astype(np.float32), "u_rand": rs.rand(n, N_IMPORTANCE).astype(np.float32)}

    def pick_threads(self):
        """Fastest thread count for this host on a 128-ray probe (all cores is not always best)."""
        if self.threads is not None:
            return self.threads
        cores = os.cpu_count() or 1
        cands = sorted({c for c in (8, 16, 32, 64, cores) if c <= cores})
        rays = blender_rays(128, 0)
        best, best_t = cores, float("inf")
        for c in cands:
            self._set_threads(c)
            self.render(rays[:16], self.replay_randoms(16, 1), 1)
            t0 = time.perf_counter()
            self.render(rays, self.replay_randoms(128, 1), 1)
            t = time.perf_counter() - t0
            if t < best_t:
                best, best_t = c, t
        self.threads = best
        self._set_threads(best)
        return best

    def _set_threads(self, c):
        if self.ref:
            self.torch.set_num_threads(c)
        else:
            try:
                from threadpoolctl import threadpool_limits
                self._limit = threadpool_limits(limits=c)
            except ImportError:
                pass

    def time_forward(self, n_rays, reps, seed=0):
        self.pick_threads()
        rays = blender_rays(n_rays, seed)
        rnd = self.replay_randoms(n_rays, seed + 1)
        self.render(rays[:32], self.replay_randoms(32, 2), 2)
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            self.render(rays, rnd, seed + 1)
            ts.append(time.perf_counter() - t0)
        t = float(np.median(ts))
        return n_rays * SAMPLES_PER_RAY / t, t

    def time_train_step(self, n_rays, reps, seed=0):
        """fwd + MSELoss + backward + Adam on the host (train.py:103-117), reference kind only."""
        if not self.ref:
            return None
        torch = self.torch
        self.pick_threads()
        rays = torch.from_numpy(blender_rays(n_rays, seed))
        tgt = torch.rand(n_rays, 3)
        params = [p for m in self.models for p in m.parameters()]
        opt = torch.optim.Adam(params, lr=5e-4)
        lossf = self.ref["MSELoss"]()
        ts = []
        for _ in range(reps + 1):
            t0 = time.perf_counter()
            opt.zero_grad()
            out = self.ref["render_rays"](self.models, self.emb, rays, N_SAMPLES, False, 1.0, 0.0, N_IMPORTANCE,
                                          1024 * 32, True, test_time=False)
            lossf(out, tgt).backward()
            opt.step()
            ts.append(time.perf_counter() - t0)
        # restore the weights the other legs use
        for m, w in zip(self.models, self.ws):
            m.load_state_dict({k: torch.from_numpy(v) for k, v in w.items()})
        return float(np.median(ts[1:]))


def workload_config(n_gpus, graph):
    return {"workload": "blender_lego_400x400 N_samples=64 N_importance=64 batch_size=1024/GPU (configs[1]; at N>1 "
                        "configs[4]'s sharded batch), render_rays perturb=1 noise_std=0 white_back test_time=False",
            "rays_per_step_per_gpu": BATCH, "global_batch": BATCH * n_gpus, "samples_per_ray": SAMPLES_PER_RAY,
            "parallelism": (f"ray-sharded dp{n_gpus}, weights replicated, one NCCL all-gather of the rendered batch "
                            f"per step" if n_gpus > 1 else "single GPU"),
            "timed_region": ("K steps in one CUDA graph, two events around the replay" if graph else
                             "eager loop, two events around K steps"),
            "l2": f"inputs larger than L2: {N_ROT} copies of the packed weights ({N_ROT * 2 * 1.09:.0f} MB read in rotation) "
                  f"and {N_ROT} ray batches, one per step; no step re-reads what the previous steps cached"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    host = HostReference()
    cores = host.pick_threads()
    n_rays = BATCH if host.kind == "reference" else 256
    for _ in range(max(min(args.warmup, 2), 1)):
        host.time_forward(n_rays, 1)
    vals = [host.time_forward(n_rays, 1, seed=i)[0] for i in range(args.steps)]
    v = float(np.median(vals))
    ms = BATCH * SAMPLES_PER_RAY / v * 1e3
    what = ("the unmodified reference (baseline/_ref: models/rendering.py render_rays + models/nerf.py, PyTorch fp32)"
            if host.kind == "reference" else "numpy port of the reference (oracle/nerf_oracle.py)")
    sample = (f"{n_rays} rays per step (64+128 samples/ray) through {what} on {cores} of {os.cpu_count()} host "
              f"threads (fastest setting probed)")
    emit(({
        "impl": "reference", "metric": "ray-samples/sec (coarse+fine)", "value": v, "unit": "ray-samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus, False),
        "cpu_baseline": {"value": v, "unit": "ray-samples/s", "cores": cores, "kind": host.kind, "sample": sample},
        "e2e": {"value": v, "unit": "ray-samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def run_b200(args):
    import torch
    import torch.distributed as dist

    import nerf_pl_b200 as nb
    from nerf_pl_b200 import _lib
    from nerf_pl_b200.sharded import render_rays_sharded

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"          # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    K = args.steps
    # randoms="kernel" seeds its draws from torch.initial_seed(): fixed, so that every run renders the same samples
    torch.manual_seed(0)

    ws = [synthetic_weights(11), synthetic_weights(12)]   # random init: there are no checkpoints
    sd = [{k: torch.from_numpy(v) for k, v in w.items()} for w in ws]

    def make_models(train=False):
        out = []
        for s in sd:
            m = nb.NeRF()
            m.load_state_dict(s)
            m = m.to(dev)
            if not train:
                m.eval().requires_grad_(False)     # inference configuration: packed once
            out.append(m)
        return out

    emb = [nb.Embedding(3, 10), nb.Embedding(3, 4)]
    model_sets = [make_models() for _ in range(N_ROT)]           # identical weights at distinct addresses
    host_rays = [torch.from_numpy(blender_rays(BATCH, 1000 * rank + i)).pin_memory() for i in range(N_ROT)]
    dev_rays = [r.to(dev) for r in host_rays]
    gather_buf = torch.empty(world * BATCH, 10, device=dev) if world > 1 else None

    ag_stream = torch.cuda.Stream() if world > 1 else None
    packed_ring = [torch.empty(BATCH, 10, device=dev) for _ in range(4)] if world > 1 else None
    overlap = {"on": world > 1 and os.environ.get("NERFB200_BENCH_AG_OVERLAP", "1") != "0", "pending": False}

    def step(i, rays=None, randoms=None):
        out = nb.render_rays(model_sets[i % N_ROT], emb, dev_rays[i % N_ROT] if rays is None else rays, N_SAMPLES, False,
                             1.0, 0.0, N_IMPORTANCE, 1024 * 32, True, test_time=False,
                             randoms="kernel" if randoms is None else randoms)
        if world > 1:      # north_star: the rendered batch is exchanged with ONE all-gather at the end of the step
            packed = packed_ring[i % 4]
            torch.cat((out["rgb_coarse"], out["depth_coarse"][:, None], out["opacity_coarse"][:, None],
                       out["rgb_fine"], out["depth_fine"][:, None], out["opacity_fine"][:, None]), 1, out=packed)
            if overlap["on"]:
                # the collective of step i runs on its own stream, behind the tail of the next step's render kernel
                # (the persistent render CTAs own all shared memory of their SM: NCCL's CTAs are placed as SMs
                # drain); join_collectives() closes the timed region
                ag_stream.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(ag_stream):
                    dist.all_gather_into_tensor(gather_buf, packed)
                overlap["pending"] = True
            else:
                dist.all_gather_into_tensor(gather_buf, packed)
        return out

    def join_collectives():
        if overlap["pending"]:
            torch.cuda.current_stream().wait_stream(ag_stream)
            overlap["pending"] = False

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_graph(fn, n_steps):
        """Capture n_steps calls of fn(i) in one CUDA graph; returns (replay callable, True) or the
        eager loop (callable, False) if capture is not possible on this box."""
        for attempt in range(2 if overlap["on"] else 1):
            try:
                g = torch.cuda.CUDAGraph()
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    fn(0)
                    join_collectives()
                torch.cuda.current_stream().wait_stream(side)
                torch.cuda.synchronize()
                with torch.cuda.graph(g):
                    for i in range(n_steps):
                        fn(i)
                    join_collectives()
                return g.replay, True
            except Exception as e:      # noqa: BLE001
                print("CUDA graph capture failed (%s): %r" % ("collective on its own stream" if overlap["on"] else
                                                              "in-stream", e), file=sys.stderr)
                overlap["pending"] = False
                torch.cuda.synchronize()
                if overlap["on"]:
                    overlap["on"] = False       # retry with the collective in the capture stream
                    continue
                break
        print("timing the eager loop", file=sys.stderr)
        if True:

            def loop():
                for i in range(n_steps):
                    fn(i)
                join_collectives()
            return loop, False

    def time_region(run):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        t0 = time.perf_counter()
        e0.record()
        run()
        e1.record()
        barrier()
        return e0.elapsed_time(e1), time.perf_counter() - t0

    with torch.no_grad():
        for i in range(max(args.warmup, N_ROT)):        # also packs every weight copy once
            step(i)
        barrier()
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        # ---- value: K steps, device-timed
        last = {}                                       # the result tensors of the last step (graph-owned when graphed)
        run, graphed = timed_graph(lambda i: last.update(step(i)) if i == K - 1 else step(i), K)
        for _ in range(2):
            run()                                       # graph warm-up replays (not timed)
        l0 = lib.nerfb200_launch_count()
        total_ms, t_wall = time_region(run)
        launches = lib.nerfb200_launch_count() - l0
        if graphed:
            launches = K                               # replayed nodes do not pass through the library's counter
        if args.dump_outputs and rank == 0:
            if world > 1:
                last["all_gather"] = gather_buf
            dump_outputs(args.dump_outputs, {k: v.cpu().numpy() for k, v in last.items()})

        # ---- kernel-only (roofline): the render kernel is the only node of a step (as in `value`: the uniform
        # numbers are Philox draws inside the kernel)
        def kstep(i):
            nb.render_rays(model_sets[i % N_ROT], emb, dev_rays[i % N_ROT], N_SAMPLES, False, 1.0, 0.0, N_IMPORTANCE,
                           1024 * 32, True, test_time=False, randoms={"seed": 1000 + i})
        krun, _ = timed_graph(kstep, K)
        krun()
        kern_total, _ = time_region(krun)
        kern_ms = kern_total / K
        # sustained: >= 1 s of back-to-back launches (power-capped behaviour)
        reps = max(1, int(1.2e3 / max(kern_total, 1e-3)))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            krun()
        e1.record()
        torch.cuda.synchronize()
        kern_ms_sustained = e0.elapsed_time(e1) / (reps * K)

        # ---- end to end through the public API with HOST buffers: nb.render_rays_host = ONE C-ABI call
        # (nerfb200_render_rays_host) that copies the pinned rays to the device, renders, copies all six
        # result tensors back to pinned memory and synchronises; the timed region is the wall clock of
        # K such calls (each returns with the result readable on the host) [+ the all-gather at N>1]
        keys = ("rgb_coarse", "depth_coarse", "opacity_coarse", "rgb_fine", "depth_fine", "opacity_fine")
        host_res = {k: torch.empty((BATCH, 3) if k.startswith("rgb") else (BATCH,)).pin_memory() for k in keys}
        packed_dev = torch.empty(BATCH, 10, device=dev)

        def e2e_step(i):
            out = nb.render_rays_host(model_sets[i % N_ROT], emb, host_rays[i % N_ROT], N_SAMPLES, False, 1.0, 0.0,
                                      N_IMPORTANCE, 1024 * 32, True, test_time=False, out=host_res, randoms="kernel")
            if world > 1:
                dist.all_gather_into_tensor(gather_buf, packed_dev)
                torch.cuda.current_stream().synchronize()
            return out
        for i in range(3):
            e2e_step(i)
        barrier()
        t0 = time.perf_counter()
        for i in range(K):
            e2e_step(i)
        e2e_ms = (time.perf_counter() - t0) * 1e3
        barrier()
        clocks = sampler.stop() if rank == 0 else None

        # ---- configs[4] inference: one 800x800 view, contiguous shards + one all-gather (strong scaling)
        img = None
        try:
            rays800 = torch.from_numpy(blender_rays(0, 7, 800, 800, pixels="all")).to(dev)
            fn = lambda r: nb.render_rays(model_sets[0], emb, r, N_SAMPLES, False, 0, 0, N_IMPORTANCE, 1024 * 32, True,
                                          test_time=True, match_reference_rng=False)
            render800 = (lambda: render_rays_sharded(fn, rays800)) if world > 1 else (lambda: fn(rays800))
            render800()
            t_img = min(time_region(render800)[0] for _ in range(2))
            img = {"rays": 640000, "ms": t_img, "value": 640000 * SAMPLES_PER_RAY / (t_img * 1e-3), "unit": "ray-samples/s",
                   "scaling": "strong", "all_gather_bytes": 640000 * 6 * 4 if world > 1 else 0,
                   "note": "test_time=True, contiguous 640000/N-ray shards, ONE all_gather_into_tensor of the packed results"}
            del rays800
        except Exception as e:      # noqa: BLE001
            img = {"error": repr(e)}

    # ---- config 2 as a TRAINING step: fused forward+loss, sm_100a backward, Adam (train.py:103-117)
    train = None
    if not args.no_train:
        try:
            tm = make_models(train=True)
            params = [p for m in tm for p in m.parameters()]
            opt = nb.FusedAdam(params, lr=5e-4)          # torch.optim.Adam's update, one launch for the 48 tensors
            tgt = [torch.rand(BATCH, 3, device=dev) for _ in range(4)]

            def tstep(i):
                opt.zero_grad(set_to_none=True)
                out = nb.render_rays_loss(tm, emb, dev_rays[i % N_ROT], tgt[i % 4], N_SAMPLES, False, 1.0, 0.0, N_IMPORTANCE,
                                          1024 * 32, True, randoms="kernel")
                out["loss"].backward()
                if world > 1:      # data-parallel training as the reference does it (DDP, train.py:174-175):
                    flat = torch._utils._flatten_dense_tensors([p.grad for p in params])    # one all-reduce of the
                    dist.all_reduce(flat)                                                    # 4.77 MB of gradients
                    flat.div_(world)
                    for p, g in zip(params, torch._utils._unflatten_dense_tensors(flat, [p.grad for p in params])):
                        p.grad = g
                opt.step()
                return out["loss"]
            for i in range(max(args.warmup, 3)):
                first = tstep(i)
            barrier()
            l0 = lib.nerfb200_launch_count()
            n_t = max(K, 10)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(n_t):
                last = tstep(i)
            e1.record()
            barrier()
            t_ms = e0.elapsed_time(e1) / n_t
            if world > 1:
                tt = torch.tensor([t_ms], device=dev)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                t_ms = float(tt)
            train = {"ms_per_step": t_ms, "value": world * BATCH * SAMPLES_PER_RAY / (t_ms * 1e-3), "unit": "ray-samples/s",
                     "steps": n_t, "kernels_per_step": (lib.nerfb200_launch_count() - l0) / n_t,
                     "includes": "pack of both weight images, fused forward + MSE loss, compositing/head/chain/wgrad/"
                                 "reduce/unfold backward kernels, Adam update (nerfb200_adam_step): every kernel of the "
                                 "step is hand-written sm_100a code of this repository",
                     "grad_allreduce": "NCCL all_reduce of the flattened gradients (4.77 MB) per step" if world > 1 else None,
                     "loss_first": float(first.detach()), "loss_last": float(last.detach()),
                     "l2": "a step streams ~3.4 GB of activations (> L2): no flush needed"}
        except Exception as e:      # noqa: BLE001
            train = {"error": repr(e)}

    # max over ranks
    t = torch.tensor([total_ms, e2e_ms, kern_ms, kern_ms_sustained, (img or {}).get("ms", 0.0)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, e2e_ms, kern_ms, kern_ms_sustained, img_ms = [float(x) for x in t.tolist()]
    if rank == 0:
        if img and "ms" in img:
            img["ms"] = img_ms
            img["value"] = 640000 * SAMPLES_PER_RAY / (img_ms * 1e-3)
        samples = BATCH * SAMPLES_PER_RAY * world * K
        value = samples / (total_ms * 1e-3)
        peak, peak_sus, peak_src = measured_peaks()
        flop = BATCH * FLOP_PER_RAY_TRAIN
        flop_x = BATCH * SAMPLES_PER_RAY * executed_flop_per_sample()
        ach = flop / (kern_ms * 1e-3) / 1e12
        traffic, pipe_pct, prof_file = ncu_profile()
        # ---- parity + CPU baseline: the reference on the host cores
        host = HostReference()
        cores = host.pick_threads()
        parity = None
        try:
            n_par = 128
            rays_np = blender_rays(BATCH, 1000 * rank)[:n_par]          # = the first rays of timed batch 0
            rnd_np = host.replay_randoms(n_par, 4321)
            ref = host.render(rays_np, rnd_np, 4321)
            with torch.no_grad():
                got = nb.render_rays(model_sets[0], emb, torch.from_numpy(rays_np).to(dev), N_SAMPLES, False, 1.0, 0.0,
                                     N_IMPORTANCE, 1024 * 32, True, test_time=False,
                                     randoms={k: torch.from_numpy(v).to(dev) for k, v in rnd_np.items()})
            dif = np.abs(got["rgb_fine"].cpu().numpy().astype(np.float64) - ref["rgb_fine"]).ravel()
            mse = float((dif ** 2).mean())
            parity = {"rgb_fine_max_abs": float(dif.max()), "rgb_fine_p99_9": float(np.percentile(dif, 99.9)),
                      "psnr_db": float(-10 * np.log10(max(mse, 1e-30))), "n_rays": n_par, "against": host.kind,
                      "rgb_coarse_max_abs": float(np.abs(got["rgb_coarse"].cpu().numpy() - ref["rgb_coarse"]).max()),
                      "bar": "rgb_fine within 1e-3 abs (north_star)"}
        except Exception as e:      # noqa: BLE001
            parity = {"error": repr(e)}
        # ---- the same check on TRAINED weights (tests/golden/trained_weights.npz: 8000 steps of this repository's own
        # training step; sharp density, large norms - where the fp16 MLP's error is largest), 1024 rays, reference only
        parity_trained = None
        tw_path = os.path.join(ROOT, "tests", "golden", "trained_weights.npz")
        if host.kind == "reference" and os.path.exists(tw_path):
            try:
                z = np.load(tw_path)
                tws = [{k[len(t) + 1:]: z[k] for k in z.files if k.startswith(t + ".")} for t in ("coarse", "fine")]
                n_tr = 1024
                rays_np = blender_rays(n_tr, 777)
                rnd_np = host.replay_randoms(n_tr, 99)
                for m, w in zip(host.models, tws):
                    m.load_state_dict({k: torch.from_numpy(v) for k, v in w.items()})
                ref = host.render(rays_np, rnd_np, 99)
                for m, w in zip(host.models, host.ws):
                    m.load_state_dict({k: torch.from_numpy(v) for k, v in w.items()})
                tm_ = []
                for w in tws:
                    m = nb.NeRF()
                    m.load_state_dict({k: torch.from_numpy(v) for k, v in w.items()})
                    tm_.append(m.to(dev).eval().requires_grad_(False))
                with torch.no_grad():
                    got = nb.render_rays(tm_, emb, torch.from_numpy(rays_np).to(dev), N_SAMPLES, False, 1.0, 0.0,
                                         N_IMPORTANCE, 1024 * 32, True, test_time=False,
                                         randoms={k: torch.from_numpy(v).to(dev) for k, v in rnd_np.items()})
                dif = np.abs(got["rgb_fine"].cpu().numpy().astype(np.float64) - ref["rgb_fine"]).max(-1)
                mse = float(((got["rgb_fine"].cpu().numpy().astype(np.float64) - ref["rgb_fine"]) ** 2).mean())
                parity_trained = {"rgb_fine_max_abs": float(dif.max()), "rgb_fine_p99": float(np.percentile(dif, 99)),
                                  "rgb_fine_p90": float(np.percentile(dif, 90)), "rgb_fine_mean": float(dif.mean()),
                                  "rays_over_1e-3": int((dif > 1e-3).sum()), "n_rays": n_tr,
                                  "psnr_db": float(-10 * np.log10(max(mse, 1e-30))), "against": "reference",
                                  "note": "per-ray max over channels; the tail is the fp16 format's (DESIGN.md section 5)"}
            except Exception as e:      # noqa: BLE001
                parity_trained = {"error": repr(e)}
        n_cpu = BATCH if host.kind == "reference" else 256
        cpu_v, cpu_t = host.time_forward(n_cpu, 3)
        cpu_train = host.time_train_step(256, 2) if host.kind == "reference" else None
        line = {
            "metric": "ray-samples/sec (coarse+fine)", "value": value, "unit": "ray-samples/s",
            "n_gpus": world, "steps": K, "warmup": args.warmup, "ms_per_step": total_ms / K,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16 (fp32 accumulate, "
            "fp32 encoding/compositing)", "data": "synthetic", "config": workload_config(world, graphed),
            "clocks": clocks,
            "e2e": {"value": samples / (e2e_ms * 1e-3), "unit": "ray-samples/s",
                    "h2d_bytes_per_step": BATCH * 8 * 4, "d2h_bytes_per_step": BATCH * 10 * 4},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s",
                         "frac": ach / peak, "traffic": traffic, "peak_source": peak_src,
                         "kernel": "render_rays_kernel", "kernel_ms": kern_ms, "flop_per_launch": flop,
                         "executed_flop_per_launch": flop_x, "frac_executed": flop_x / (kern_ms * 1e-3) / 1e12 / peak,
                         "kernel_ms_sustained": kern_ms_sustained,
                         "frac_sustained": flop / (kern_ms_sustained * 1e-3) / 1e12 / peak_sus,
                         "peak_sustained": peak_sus,
                         "tensor_pipe_active_pct": pipe_pct, "ncu_capture": prof_file},
            "cpu_baseline": {"value": cpu_v, "unit": "ray-samples/s", "cores": cores, "kind": host.kind,
                             "sample": f"{n_cpu} rays of the same workload, 3 reps, median {cpu_t:.2f} s, on {cores} of "
                                       f"{os.cpu_count()} host threads (fastest setting probed)",
                             "train_step_s_256_rays": cpu_train},
            "parity": parity,
            "parity_trained_weights": parity_trained,
            "train": train,
            "image_800": img,
            "collective": (("NCCL all_gather_into_tensor, %d B per rank per step" % (BATCH * 40)) +
                           (", enqueued on its own stream inside the graph: the collective of step i runs behind the tail "
                            "of step i+1's render kernel; the last one is joined before the closing event"
                            if overlap["on"] else ", in the step's stream")) if world > 1 else None,
            "wall_s_timed_region": t_wall,
        }
        emit(line)
    if world > 1:
        # Leave without relying on interpreter / C++ teardown: at N = 8 (r02, NVLS communicator, collectives captured
        # in CUDA graphs) the process printed its line and then sat in teardown until the box's limit killed it.
        # Order: drop the graphs that hold NCCL nodes (their destruction releases NCCL's graph registrations), drain
        # the device, give destroy_process_group a bounded chance (it releases the GIL), then leave with os._exit -
        # through the atexit hooks only if the process group is really gone (torch registers an exit-time NCCL abort
        # that could block on a half-destroyed group).  The result line is already on the original stdout.  Last
        # resort, independent of the GIL: faulthandler's watchdog thread ends the process 240 s after this point.
        import faulthandler
        import gc
        faulthandler.dump_traceback_later(240, exit=True)
        barrier()                      # the other ranks wait here for rank 0's host-side legs: teardown starts together
        run = krun = None
        gc.collect()
        torch.cuda.synchronize()
        clean = _bounded(dist.destroy_process_group, 20.0, dev)
        _hard_exit(0, run_atexit=clean, device=dev)


def _bounded(fn, seconds, device=None):
    """Run fn() on a daemon thread, wait at most `seconds`; True if it finished.  `device`: the CUDA device to make
    current in that thread first (the current device is thread-local; a fresh thread would otherwise touch device 0)."""
    def target():
        if device is not None:
            import torch
            torch.cuda.set_device(device)
        fn()
    t = threading.Thread(target=target, daemon=True)
    t.start()
    t.join(seconds)
    return not t.is_alive()


def _hard_exit(code, run_atexit=True, device=None):
    import atexit
    if run_atexit:
        _bounded(atexit._run_exitfuncs, 10.0, device)
    try:
        sys.stdout.flush()
        sys.stderr.flush()
    except Exception:      # noqa: BLE001
        pass
    os._exit(code)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write each array as out_dir/<name>.npy (float32 or float64), so that two builds can be compared output
    for output on the same seeded inputs."""
    for name, a in arrays.items():
        if a.dtype not in (np.float32, np.float64):
            raise TypeError(f"{name}: dtype {a.dtype} is not float32 / float64")
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"outputs take {total} bytes, more than the {DUMP_LIMIT_BYTES} allowed")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


_JSON_FD = None


def emit(obj):
    """The ONE JSON line goes to the process's original stdout; everything else that libraries
    print on fd 1 (e.g. NCCL's version banner) has been redirected to stderr by main()."""
    data = (json.dumps(obj) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    global _JSON_FD
    sys.dont_write_bytecode = True      # the project's modules are imported later; no __pycache__ in the tree
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-train", action="store_true", help="skip the training-step leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the result tensors of the last one to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
