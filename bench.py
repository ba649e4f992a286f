#!/usr/bin/env python
"""bench.py -- Mrays/s of the tracing hot path (forward + backward) on the BASELINE.json
headline workload: synthetic 1,048,576-point foam, one 1920x1080 frame, Q = 2 depth
quantiles, sh_degree 3, fp32 (config 4; SURVEY.md §8d).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over the frame: scene re-layout (points/attributes
change every training step, so mirrors are rebuilt once per step), trace_forward,
trace_backward (+ one all-reduce of the per-point gradient accumulator when N > 1).
`value`: inputs resident in HBM.  `e2e`: the same step through the public autograd op with
the step's inputs in pinned HOST memory (H2D inside the timed region) and the loss read back.
Rank 0 prints ONE JSON line.  The oracle is used only by the cpu_baseline leg and by
--impl reference (which times the reference's OWN CUDA kernels from oracle/_ref).
--dump-outputs DIR writes what the last timed step returned (see dump_outputs) so that two builds can be compared.
The run writes nothing into the source tree (which may be read-only): the foam cache lives under the system's
temporary directory.
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys
import tempfile
import time

sys.dont_write_bytecode = True

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "Mrays/s fwd+bwd @1080p, 1M-point foam"
CAMERA_POS = (2.5, 2.5, 2.5)
FOV = 0.9


# ----------------------------------------------------------------------------- workload
def load_or_build_foam(num_points: int, log):
    """Delaunay adjacency costs ~35 s/Mpoint on one core (and on an N-GPU box every GPU is charged while rank 0
    builds it).  Two caches: the full foam under the temporary directory (machine-local), and the packed ADJACENCY
    only under foam_cache/ (17 MB per Mpoint; git-ignored, read if present) -- points and attributes are regenerated
    from the seed in seconds."""
    from radfoam_b200 import foam

    cache_dir = os.path.join(tempfile.gettempdir(), f"radfoam_b200_bench_cache_{os.getuid()}")
    path = os.path.join(cache_dir, f"foam_{num_points}.npz")
    if os.path.exists(path):
        z = np.load(path)
        f = foam.Foam(z["points"], z["attributes"], z["adjacency"], z["offsets"], 3)
        log(f"foam cache hit: {path}")
        return f
    t0 = time.time()
    adj_path = next((q for q in (os.path.join(ROOT, d, f"adjacency_{num_points}.npz")
                                 for d in ("foam_cache", "foam_cache_big")) if os.path.exists(q)), None)
    if adj_path:
        z = np.load(adj_path)
        f = foam.scene_foam(num_points, sh_degree=3, adjacency=foam.unpack_adjacency(z["counts"], z["delta"]))
        log(f"foam from the shipped adjacency: {f.num_points} points, E={f.adjacency.size}, {time.time() - t0:.1f} s")
        return f
    f = foam.scene_foam(num_points, sh_degree=3)
    log(f"foam built: {f.num_points} points, E={f.adjacency.size}, {time.time() - t0:.1f} s")
    try:
        os.makedirs(cache_dir, exist_ok=True)
        np.savez(path + ".tmp.npz", points=f.points, attributes=f.attributes, adjacency=f.adjacency,
                 offsets=f.offsets)
        os.replace(path + ".tmp.npz", path)
        os.sync()  # finish the write-back now, not under the timed region
    except OSError:
        pass
    return f


def pack_foam_adjacency(num_points: int):
    """python -c 'import bench; bench.pack_foam_adjacency(N)': write foam_cache/adjacency_N.npz (run where CPU time
    is free, before a multi-GPU call)."""
    from radfoam_b200 import foam

    f = load_or_build_foam(num_points, print)
    os.makedirs(os.path.join(ROOT, "foam_cache"), exist_ok=True)
    np.savez_compressed(os.path.join(ROOT, "foam_cache", f"adjacency_{num_points}.npz"),
                        **foam.pack_adjacency(f.adjacency, f.offsets))


def workload_name(f, width: int, height: int) -> str:
    """Identical in both arms (the driver compares the strings)."""
    name = {(1_048_576, 1920, 1080): "config4", (2_097_152, 1920, 1080): "config3-sized",
            (4_194_304, 3840, 2160): "config5-sized", (524_288, 1920, 1080): "config2-sized"}.get(
        (f.num_points, width, height), "custom")
    return (f"{name}: synthetic foam {f.num_points} points (E={f.adjacency.size}), {width}x{height} frame, "
            "Q=2, sh_degree 3, fwd+bwd")


def make_frame(f, width: int, height: int):
    from radfoam_b200 import foam

    rays = foam.pinhole_rays(width, height, CAMERA_POS, fov=FOV)
    start = np.full((height, width), foam.nearest_point(f.points, CAMERA_POS), dtype=np.uint32)
    rng = np.random.default_rng(4)
    # training passes two sorted-descending uniform quantiles per ray (train.py:176-180)
    dq = np.sort(rng.uniform(0.0, 1.0, size=(height, width, 2)).astype(np.float32), axis=-1)[..., ::-1].copy()
    grad_rgba = rng.normal(size=(height, width, 4)).astype(np.float32)
    grad_depth = (rng.normal(size=(height, width, 2)) * 1e-4).astype(np.float32)
    target = rng.uniform(0.0, 1.0, size=(height, width, 4)).astype(np.float32)
    return dict(rays=rays, start=start, dq=dq, grad_rgba=grad_rgba, grad_depth=grad_depth, target=target)


DUMP_RAYS, DUMP_POINTS = 131_072, 131_072  # sampled rows: ~36 MB for the headline workload


def sample_outputs(outputs: dict, ray_shape: tuple, num_points: int) -> dict:
    """What one step returned, as float32 / float64 host arrays of at most DUMP_RAYS rays and DUMP_POINTS points.  The
    rows are a fixed, seeded sample (the same for every run with the same arguments); their indices are included as
    ray_index and point_index.  ray_index indexes the flattened per-ray batch the step traced: the whole image on one
    GPU; with --gpus N > 1, rank 0 writes the dump and its batch is rank 0's shard (its interleaved 8-row bands), while
    the gradients, reduced over all ranks, are the whole step's.  Integer outputs are stored as float64, which holds
    uint32 exactly.  ray_grad is left out: the path allocates it but never writes it."""
    import torch

    out = {}
    for name, t in sorted(outputs.items()):
        if name == "ray_grad" or t is None:
            continue
        per_ray = tuple(t.shape[:len(ray_shape)]) == tuple(ray_shape)
        assert per_ray or t.shape[0] == num_points, (name, tuple(t.shape))
        rows = t.reshape(-1, *t.shape[len(ray_shape):]) if per_ray else t
        key, limit = ("ray_index", DUMP_RAYS) if per_ray else ("point_index", DUMP_POINTS)
        if key not in out:
            count = rows.shape[0]
            idx = np.arange(count) if count <= limit else np.sort(
                np.random.default_rng(1).choice(count, size=limit, replace=False))
            out[key] = idx.astype(np.float64)
        rows = rows.detach().index_select(0, torch.from_numpy(out[key].astype(np.int64)).to(rows.device))
        if rows.is_floating_point():
            out[name] = rows.float().cpu().numpy()
        else:
            out[name] = rows.to(torch.int64).cpu().numpy().astype(np.float64)
    return out


def dump_outputs(directory: str, arrays: dict):
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU during the timed region (NVML, every few
    milliseconds from a thread: the timed region of a short run is only tens of milliseconds)."""

    def __init__(self, index: int, period_s: float = 0.004):
        import threading

        self.samples, self.reasons, self.max_mhz, self.err = [], set(), None, None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml

            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            names = {"hw_slowdown": getattr(pynvml, "nvmlClocksEventReasonHwSlowdown", 0x8),
                     "hw_thermal_slowdown": getattr(pynvml, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                     "sw_thermal_slowdown": getattr(pynvml, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                     "sw_power_cap": getattr(pynvml, "nvmlClocksEventReasonSwPowerCap", 0x4)}
            get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                getattr(pynvml, "nvmlDeviceGetCurrentClocksThrottleReasons")

            def loop():
                while not self._stop.is_set():
                    try:
                        self.samples.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                        mask = int(get_reasons(h))
                        for n, bit in names.items():
                            if mask & bit:
                                self.reasons.add(n)
                    except Exception as e:  # noqa: BLE001
                        self.err = repr(e)
                        return
                    self._stop.wait(period_s)

            self._thread = threading.Thread(target=loop, daemon=True)
            self._thread.start()
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def stop(self) -> dict:
        self._stop.set()
        if self._thread is not None:
            self._thread.join(timeout=2)
        out = {"sm_mhz": float(np.median(self.samples)) if self.samples else None,
               "sm_max_mhz": self.max_mhz, "samples": len(self.samples), "reasons": sorted(self.reasons)}
        if self.err:
            out["sampler_error"] = self.err
        return out


# ----------------------------------------------------------------------------- helpers
class InputPrefetcher:
    """Host -> device feed for the e2e legs of BOTH arms: step i's inputs are copied from pinned
    host memory on a private copy stream into one of two pre-allocated device buffer sets, one
    step ahead of their use -- what the reference's BatchFetcher does
    (src/utils/batch_fetcher.cpp:44-117: cuMemcpyHtoDAsync on its own stream, ring of batches)."""

    def __init__(self, host, keys, dev):
        import torch

        self.torch, self.host, self.keys, self.dev = torch, host, keys, dev
        self.stream = torch.cuda.Stream(device=dev)
        self.bufs = [{k: torch.empty_like(host[k], device=dev) for k in keys} for _ in range(2)]
        self.free = [None, None]  # event: the compute that last read this buffer set has finished

    def enqueue(self, i):
        torch = self.torch
        b = i % 2
        with torch.cuda.stream(self.stream):
            if self.free[b] is not None:
                self.stream.wait_event(self.free[b])
            t0 = torch.cuda.Event(enable_timing=True)
            t0.record(self.stream)
            for k in self.keys:
                self.bufs[b][k].copy_(self.host[k], non_blocking=True)
            ev = torch.cuda.Event(enable_timing=True)
            ev.record(self.stream)
        self.last = (t0, ev)
        return self.bufs[b], ev

    def last_copy_ms(self):
        """Duration of the most recent H2D batch on the copy stream (diagnostic: PCIe health)."""
        t0, t1 = self.last
        t1.synchronize()
        return float(t0.elapsed_time(t1))

    def release(self, i):
        self.free[i % 2] = self.torch.cuda.current_stream(self.dev).record_event()


def measured_peak_hbm():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured"
    except (OSError, KeyError, ValueError):
        return 6650.0, "fallback"


def algorithmic_bytes(num_steps: int, num_rays: int, mean_degree: float, attr_dim: int, q: int):
    """Bytes each ray kernel has to touch under SURVEY.md §8(d)'s no-reuse gather model, fp32
    attributes (s = 4), stated per ray-step and per ray (DESIGN.md §4):
      forward  (records the tape): offsets 8 + faces 8*deg + neighbour 4 + next point/density 16
                                   + attribute row s*(A-1) + tape record 8
      backward (replays the tape): tape record 8 + next point/density 16 + attribute row s*(A-1)
                                   + gradient row read-modify-write counted once s*A + position
                                   gradient 12
    The reference's re-walk backward would be forward + s*A + 12 = 551 B; replaying the tape
    removes the face and offset reads from the backward."""
    s = 4
    b_f = 8 + 8 * mean_degree + 4 + 16 + s * (attr_dim - 1) + 8
    b_b = 8 + 16 + s * (attr_dim - 1) + s * attr_dim + 12
    fixed_f = 24 + 4 + 4 * s + 4 + q * 12 + 8
    fixed_b = 24 + 4 + 4 * s + 4 * s + q * 12 + 8
    return (num_steps * b_f + num_rays * fixed_f, num_steps * b_b + num_rays * fixed_b, b_f, b_b)


def compulsory_bytes(num_steps: int, num_rays: int, cells: int, mean_degree: float, attr_dim: int, q: int):
    """DRAM bytes one launch cannot avoid (SURVEY.md §8d's compulsory bound): unique cells x row bytes + the
    tape + per-ray inputs/outputs.  forward (records): per touched cell 16 (cell) + 8 (offsets) + 12*deg
    (face + neighbour rows) + 4*(A-1) (SH row); 8 per ray-step (tape write); per ray 24 + 4 + 16 + 4 + 20 q + 8.
    backward (replays): per touched cell 16 + 4*(A-1) + 2 * 4 * grad_row (accumulator read-modify-write);
    8 per ray-step (tape read); per ray 24 + 4 + 16 + 16 + 20 q + 8."""
    grad_row = ((attr_dim - 1 + 3) // 4) * 4 + 4
    fwd = cells * (16 + 8 + 12 * mean_degree + 4 * (attr_dim - 1)) + 8 * num_steps + num_rays * (56 + 20 * q)
    bwd = cells * (16 + 4 * (attr_dim - 1) + 8 * grad_row) + 8 * num_steps + num_rays * (68 + 20 * q)
    return {"forward_kernel": float(fwd), "backward_kernel": float(bwd)}


def dist_setup(gpus: int):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(0)
    if gpus != world:
        if rank == 0:
            print(f"bench.py: --gpus {gpus} but WORLD_SIZE={world}; launch with torch.distributed.run",
                  file=sys.stderr)
        gpus = world
    return rank, world, local


def max_over_ranks(ms: float, world: int) -> float:
    if world == 1:
        return ms
    import torch
    import torch.distributed as dist

    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def barrier(world: int):
    import torch

    if world > 1:
        import torch.distributed as dist

        dist.barrier()
    torch.cuda.synchronize()


def broadcast_foam(f, rank: int, world: int, num_points: int, log):
    """Rank 0 builds (or loads) the foam; the others receive it over NCCL."""
    import torch
    import torch.distributed as dist

    from radfoam_b200 import foam

    if world == 1:
        return load_or_build_foam(num_points, log)
    if rank == 0:
        f = load_or_build_foam(num_points, log)
        meta = torch.tensor([f.num_points, f.adjacency.size], dtype=torch.int64, device="cuda")
    else:
        meta = torch.zeros(2, dtype=torch.int64, device="cuda")
    dist.broadcast(meta, 0)
    n, e = int(meta[0]), int(meta[1])
    arrays = []
    for name, shape, dt in (("points", (n, 3), np.float32), ("attributes", (n, 49), np.float32),
                            ("adjacency", (e,), np.int32), ("offsets", (n + 1,), np.int32)):
        if rank == 0:
            t = torch.from_numpy(getattr(f, name).view(dt) if dt == np.int32 else getattr(f, name)).cuda()
        else:
            t = torch.empty(shape, dtype=torch.float32 if dt == np.float32 else torch.int32, device="cuda")
        dist.broadcast(t, 0)
        arrays.append(t.cpu().numpy())
    return foam.Foam(arrays[0], arrays[1], arrays[2].view(np.uint32), arrays[3].view(np.uint32), 3)


# ----------------------------------------------------------------------------- ours
def run_ours(args):
    import torch

    import radfoam_b200
    from radfoam_b200 import pipeline as rp
    from radfoam_b200 import sharded

    rank, world, local = dist_setup(args.gpus)
    log = (lambda m: print(f"[bench] {m}", file=sys.stderr, flush=True)) if rank == 0 else (lambda m: None)
    dev = torch.device("cuda", local)
    f = broadcast_foam(None, rank, world, args.points, log)
    frame = make_frame(f, args.width, args.height)
    H, W = args.height, args.width
    R_total = H * W

    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    # scene parameters are trainable (requires_grad), as in train.py: this is what makes the
    # forward record the walk tape for the backward of the same step
    points, attrs = d(f.points).requires_grad_(True), d(f.attributes).requires_grad_(True)
    adj, off = d(f.adjacency), d(f.offsets)
    pipe = radfoam_b200.create_pipeline(3, "float32")
    tracer = sharded.ShardedTracer(pipe)
    if args.emulate_shard and world == 1:
        # profiling aid: trace rank 0's shard of an N-way split on ONE GPU (no collective) -- the per-GPU
        # work of the N-GPU run, e.g. for an ncu capture at the N = 8 shard size
        tracer.rank, tracer.world = 0, int(args.emulate_shard)

    # this rank's shard of every per-ray tensor (interleaved 8-row bands)
    host = {k: torch.from_numpy(v) for k, v in frame.items()}
    shard_host = {k: tracer.shard(v, image=True).contiguous().pin_memory() for k, v in host.items()}
    if args.emulate_shard and world == 1:
        tracer.rank, tracer.world = 0, 1  # shards are cut; from here on behave as a single rank
    dv = {k: v.to(dev) for k, v in shard_host.items()}
    R_local = dv["rays"].shape[0] * dv["rays"].shape[1]
    if args.emulate_shard and world == 1:
        R_total = R_local  # the line then describes the shard alone

    def step_device():
        pipe.invalidate_cache()  # new parameter values every training step
        fwd = tracer.trace_forward(points, attrs, adj, off, dv["rays"], dv["start"], depth_quantiles=dv["dq"])
        bwd = tracer.trace_backward(points, attrs, adj, off, dv["rays"], dv["start"], fwd["rgba"],
                                    dv["grad_rgba"], dv["dq"], fwd["depth_indices"], dv["grad_depth"],
                                    scrub_nonfinite=True)
        return fwd, bwd

    pts_p = points.detach().clone().requires_grad_(True)
    attrs_p = attrs.detach().clone().requires_grad_(True)

    fetch = InputPrefetcher(shard_host, ("rays", "start", "dq", "target"), dev)

    phase_names = ("enqueue_h2d", "forward_call", "loss_ops", "backward_call", "loss_readback")
    e2e_phases = []   # per step: host milliseconds spent in each phase
    e2e_cpu = []      # per step: CPU time of the main thread (a gap to the wall time = descheduled / blocked)
    e2e_gpu_ev = []   # per step: CUDA events around the step's GPU work

    def step_e2e(batch, ev, ph):
        t0 = time.perf_counter()
        e_a = torch.cuda.Event(enable_timing=True)
        torch.cuda.current_stream(dev).wait_event(ev)
        e_a.record()
        pipe.invalidate_cache()
        pts_p.grad = None
        attrs_p.grad = None
        rgba, depth, _, _ = sharded.ShardedTraceRays.apply(tracer, pts_p, attrs_p, adj, off, batch["rays"],
                                                           batch["start"], batch["dq"], False)
        t1 = time.perf_counter()
        # train.py:187-204 shape: colour loss + depth-quantile regulariser (sums: shards add up)
        loss = (((rgba - batch["target"]) ** 2).sum() / R_total
                + 1e-4 * (depth[..., 0] - depth[..., 1]).abs().sum() / R_total)
        t2 = time.perf_counter()
        loss.backward()
        e_b = torch.cuda.Event(enable_timing=True)
        e_b.record()
        t3 = time.perf_counter()
        ph[1:4] = [(t1 - t0) * 1e3, (t2 - t1) * 1e3, (t3 - t2) * 1e3]
        e2e_gpu_ev.append((e_a, e_b))
        return loss

    e2e_step_wall = []

    def run_e2e(steps):
        """K steps; every step's H2D copy is issued inside this region, one step ahead of its use
        (copy of step i+1 overlaps the kernels of step i); the loss is read back every step."""
        nxt = fetch.enqueue(0)
        last = 0.0
        e2e_step_wall.clear()
        e2e_phases.clear()
        e2e_cpu.clear()
        e2e_gpu_ev.clear()
        for i in range(steps):
            t_step = time.perf_counter()
            c_step = time.thread_time()
            ph = [0.0] * 5
            batch, ev = nxt
            if i + 1 < steps:
                nxt = fetch.enqueue(i + 1)
            ph[0] = (time.perf_counter() - t_step) * 1e3
            loss = step_e2e(batch, ev, ph)
            t_r = time.perf_counter()
            last = float(loss.item())  # D2H read of the step's result
            ph[4] = (time.perf_counter() - t_r) * 1e3
            fetch.release(i)
            e2e_step_wall.append((time.perf_counter() - t_step) * 1e3)
            e2e_cpu.append((time.thread_time() - c_step) * 1e3)
            e2e_phases.append(ph)
        return last

    # --- warm-up (also gives the work counters)
    for _ in range(max(args.warmup, 3)):
        fwd, bwd = step_device()
    torch.cuda.synchronize()
    nint_local = fwd["num_intersections"].to(torch.int64)
    steps_local = int(nint_local.sum().item())
    n_mean, n_max = float(nint_local.float().mean().item()), int(nint_local.max().item())
    # cells this rank's rays composite at least once (for the compulsory-traffic bound of the roofline)
    with torch.no_grad():
        contrib = pipe.trace_forward(points, attrs, adj, off, dv["rays"], dv["start"],
                                     return_contribution=True)["contribution"]
    cells_touched = int((contrib > 0).sum().item())
    del contrib

    # --- timed region: exactly K steps, events on the launching stream, max over ranks
    pipe.set_profiling(True)
    rp.reset_launch_count()
    sampler = ClockSampler(local) if rank == 0 else None
    barrier(world)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fwd_ms, bwd_ms = [], []
    ev0.record()
    for _ in range(args.steps):
        last_step = step_device()
        if args.kernel_times:
            fwd_ms.append(pipe.last_kernel_ms("forward"))
            bwd_ms.append(pipe.last_kernel_ms("backward"))
    ev1.record()
    barrier(world)
    total_ms = max_over_ranks(ev0.elapsed_time(ev1), world)
    dumped = (sample_outputs(dict(last_step[0], **last_step[1]), dv["rays"].shape[:-1], points.shape[0])
              if args.dump_outputs else None)
    del last_step
    clocks = sampler.stop() if sampler else None
    launches = rp.launch_count()
    # per-phase durations from a separate short pass (events between the phases would serialise the timed loop)
    phase_rows, exchange_rows = [], []
    tracer.profile_reduce = True
    for _ in range(3):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        pipe.invalidate_cache()
        ev[0].record()
        fwd = tracer.trace_forward(points, attrs, adj, off, dv["rays"], dv["start"], depth_quantiles=dv["dq"])
        ev[1].record()
        acc, _ = pipe.trace_backward_accumulate(points, attrs, adj, off, dv["rays"], dv["start"], fwd["rgba"],
                                                dv["grad_rgba"], dv["dq"], fwd["depth_indices"], dv["grad_depth"])
        ev[2].record()
        tracer.reduce_and_finalize(points.shape[0], dev, True, acc)
        ev[3].record()
        torch.cuda.synchronize()
        kf, kb = pipe.last_kernel_ms("forward"), pipe.last_kernel_ms("backward")
        if not args.kernel_times:
            fwd_ms.append(kf)
            bwd_ms.append(kb)
        phase_rows.append([ev[0].elapsed_time(ev[1]) - kf, kf, ev[1].elapsed_time(ev[2]) - kb, kb,
                           ev[2].elapsed_time(ev[3])])
        if tracer.last_reduce_ms():
            exchange_rows.append(tracer.last_reduce_ms())
    tracer.profile_reduce = False
    phase_names_dev = ("relayout_and_tape_setup", "forward_kernel", "accumulator_zero_fill", "backward_kernel",
                       "grad_reduce_and_finalize")
    phases_ms = {n: round(float(np.median([r[j] for r in phase_rows])), 4) for j, n in enumerate(phase_names_dev)}
    if exchange_rows:
        phases_ms["grad_reduce_and_finalize_parts"] = {k: round(float(np.median([r[k] for r in exchange_rows])), 4)
                                                       for k in exchange_rows[0]}
    if world > 1:  # every rank's phases: the step is as long as its slowest rank
        import torch.distributed as dist

        mine = torch.tensor([[r[j] for j in range(5)] for r in phase_rows], dtype=torch.float64, device=dev).median(0).values
        every = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(every, mine)
        table = torch.stack(every).cpu().numpy()
        phases_ms["per_rank"] = {n: [round(float(x), 3) for x in table[:, j]] for j, n in enumerate(phase_names_dev)}
    pipe.set_profiling(False)
    ms_per_step = total_ms / args.steps

    # --- e2e: host buffers -> public autograd op -> loss back on the host
    run_e2e(max(args.warmup, 3))
    # the e2e loop synchronises every step, so host hiccups are exposed: keep the cyclic collector (the
    # foam build leaves a large heap) out of the timed region
    gc.collect()
    gc.freeze()
    if not os.environ.get("RFB_BENCH_GC_ON"):
        gc.disable()
    barrier(world)
    mem0 = torch.cuda.memory_stats(dev)
    lib0 = rp.device_alloc_counts()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    loss_val = run_e2e(args.steps)
    e1.record()
    barrier(world)
    gc.enable()
    mem1 = torch.cuda.memory_stats(dev)
    lib1 = rp.device_alloc_counts()
    e2e_ms = max_over_ranks(e0.elapsed_time(e1), world) / args.steps
    e2e_steps = [round(x, 2) for x in e2e_step_wall]
    h2d = sum(shard_host[k].numel() * shard_host[k].element_size() for k in ("rays", "start", "dq", "target"))
    h2d_ms = fetch.last_copy_ms()
    wall = np.array(e2e_step_wall)
    slow = [int(i) for i in np.nonzero(wall > 1.3 * np.median(wall))[0]]
    ph = np.array(e2e_phases)
    gpu_ms = np.array([a.elapsed_time(b) for a, b in e2e_gpu_ev])
    e2e_diag = {
        "step_wall_ms": {"min": float(wall.min()), "median": float(np.median(wall)), "max": float(wall.max())},
        "steps_over_1p3x_median": slow,
        "phase_ms_median": {n: round(float(np.median(ph[:, j])), 3) for j, n in enumerate(phase_names)},
        "phase_ms_max": {n: round(float(ph[:, j].max()), 3) for j, n in enumerate(phase_names)},
        "slow_steps": [{"step": i, "wall_ms": round(float(wall[i]), 2), "cpu_ms": round(float(e2e_cpu[i]), 2),
                        "gpu_ms": round(float(gpu_ms[i]), 2),
                        "phases": {n: round(float(ph[i, j]), 2) for j, n in enumerate(phase_names)}}
                       for i in slow[:8]],
        "gpu_step_ms": {"min": float(gpu_ms.min()), "median": float(np.median(gpu_ms)), "max": float(gpu_ms.max())},
        "torch_device_allocs": int(mem1.get("num_device_alloc", 0) - mem0.get("num_device_alloc", 0)),
        "torch_device_frees": int(mem1.get("num_device_free", 0) - mem0.get("num_device_free", 0)),
        "torch_alloc_retries": int(mem1.get("num_alloc_retries", 0) - mem0.get("num_alloc_retries", 0)),
        "torch_reserved_bytes": int(mem1.get("reserved_bytes.all.current", 0)),
        "torch_reserved_growth_bytes": int(mem1.get("reserved_bytes.all.current", 0)
                                           - mem0.get("reserved_bytes.all.current", 0)),
        "lib_device_allocs": lib1[0] - lib0[0], "lib_device_frees": lib1[1] - lib0[1],
        "gc": "on" if os.environ.get("RFB_BENCH_GC_ON") else "frozen+disabled",
    }

    # --- e2e again, the step captured in a CUDA graph (the path is graph-capturable: SURVEY.md §7).  Same work:
    # H2D copy of the step's inputs from pinned memory on the copy stream, the public autograd op + the loss +
    # backward (now one graph launch instead of ~40 kernel launches and the autograd dispatch), loss read back
    # every step.  One graph per input buffer set.  All ranks must agree on whether it worked.
    graph_e2e = None
    if os.environ.get("RFB_BENCH_E2E_GRAPH", "1") != "0":
        graph_e2e = run_e2e_graph(torch, dev, world, args, fetch, pipe, tracer, sharded, pts_p, attrs_p, adj, off,
                                  R_total, barrier, max_over_ranks, log)

    if rank != 0:
        return
    # --- roofline of the dominant kernel (the backward ray kernel), this rank's launch
    peak, peak_src = measured_peak_hbm()
    mean_deg = f.adjacency.size / f.num_points
    bytes_f, bytes_b, b_f, b_b = algorithmic_bytes(steps_local, R_local, mean_deg, 49, 2)
    k_fwd, k_bwd = float(np.mean(fwd_ms)), float(np.mean(bwd_ms))
    dominant = "backward_kernel" if k_bwd >= k_fwd else "forward_kernel"
    gather_bytes, dom_ms = (bytes_b, k_bwd) if k_bwd >= k_fwd else (bytes_f, k_fwd)
    comp = compulsory_bytes(steps_local, R_local, cells_touched, mean_deg, 49, 2)
    dom_bytes = comp[dominant]
    achieved = dom_bytes / (dom_ms * 1e-3) / 1e9
    limits = {}
    lpath = os.path.join(ROOT, "profiles", "kernel_limits.json")
    if os.path.exists(lpath):
        try:
            limits = json.load(open(lpath))
        except (OSError, ValueError):
            limits = {}
    lim = limits.get(dominant, {})
    traffic = lim.get("dram_bytes_per_launch") if world == 1 and not args.emulate_shard else None
    cpu = cpu_baseline(f, frame, log) if not args.no_cpu_baseline else None
    try:
        tape = pipe.tape_status()
    except RuntimeError:
        tape = None

    line = {
        "metric": METRIC, "value": R_total / (ms_per_step * 1e-3) / 1e6, "unit": "Mrays/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "impl": "ours",
        "config": {"workload": workload_name(f, W, H),
                   "step": "scene re-layout (parameters change every training step) + trace_forward + "
                           "trace_backward" + (f"; rank 0's shard of a {args.emulate_shard}-way ray split only"
                                               if args.emulate_shard else ""),
                   "rays": R_total, "mean_cells_per_ray": n_mean, "max_cells_per_ray": n_max,
                   "parallelism": f"ray-sharded x{world} (8-row bands), {tracer.reduction_name()} of the [N,52] fp32 "
                                  "gradient accumulator"
                   if world > 1 else "single GPU",
                   "l2": "scene working set (417 MB) larger than L2 (126 MB); no explicit flush"},
        "clocks": clocks,
        "e2e": {"value": R_total / (e2e_ms * 1e-3) / 1e6, "unit": "Mrays/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 4, "loss": loss_val,
                "h2d_ms_per_step": h2d_ms, "h2d_overlapped": True, "host_wall_ms_each_step": e2e_steps,
                "mode": "eager", "diag": e2e_diag},
        "gpu_launches": int(launches),
        "kernels_ms": {"forward_kernel": k_fwd, "backward_kernel": k_bwd},
        "walk_tape": tape,
        "phases_ms": phases_ms,
        "roofline": {"bound": "hbm", "kernel": dominant, "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "peak_source": peak_src, "traffic": traffic,
                     "algorithmic_bytes_per_launch": dom_bytes,
                     "algorithmic_model": "compulsory DRAM bytes: every ray-step reads (forward: writes) its 8-byte "
                                          "tape record once; every cell the launch composites is fetched once "
                                          "(16 B cell + 192 B SH row; forward also its face row) and its 208 B "
                                          "gradient row is read and written once; per-ray inputs/outputs once",
                     "ray_steps_per_launch": steps_local, "cells_touched": cells_touched,
                     "dram_frac": (traffic / (dom_ms * 1e-3) / 1e9 / peak) if traffic else None,
                     "traffic_over_algorithmic": (traffic / dom_bytes) if traffic else None,
                     # what actually limits the kernel (ncu --set full of the same command, profiles/):
                     "binding_limit": lim.get("binding_limit"),
                     "binding_frac": lim.get("binding_frac"),
                     "speed_of_light": lim.get("speed_of_light"),
                     "source": limits.get("source"),
                     "effective_gather_gbs": gather_bytes / (dom_ms * 1e-3) / 1e9,
                     "note": "NOT an HBM-bound kernel: achieved/frac state how little of the HBM roofline the "
                             "path needs (the cell working set is re-used from L1/L2; most DRAM bytes are the "
                             "walk tape). The limit that binds is binding_limit (fraction of its peak = "
                             "binding_frac). effective_gather_gbs is round 1's no-reuse gather model "
                             "(bytes every ray-step would fetch without any cache), kept for continuity; it "
                             "is not a bound."},
        "cpu_baseline": cpu,
    }
    if graph_e2e and graph_e2e.get("ok"):
        # the headline end-to-end figure is the better-supported way to run the same step; the eager loop stays
        line["e2e_eager"] = dict(line["e2e"])
        line["e2e"].update({"value": R_total / (graph_e2e["ms_per_step"] * 1e-3) / 1e6,
                            "ms_per_step": graph_e2e["ms_per_step"], "loss": graph_e2e["loss"],
                            "mode": "cuda_graph (one captured graph per input buffer set: H2D on the copy stream, "
                                    "graph replay, loss.item())",
                            "host_wall_ms_each_step": graph_e2e["wall_ms"],
                            "loss_matches_eager": graph_e2e["loss"] == loss_val})
        line["e2e"]["diag"] = {"step_wall_ms": graph_e2e["wall_stats"], "eager": e2e_diag}
    elif graph_e2e:
        line["e2e"]["cuda_graph_unavailable"] = graph_e2e.get("error")
    if dumped is not None:
        dump_outputs(args.dump_outputs, dumped)
    print(json.dumps(line), flush=True)


def run_e2e_graph(torch, dev, world, args, fetch, pipe, tracer, sharded, pts_p, attrs_p, adj, off, R_total, barrier,
                  max_over_ranks, log):
    """The e2e step of run_ours captured into CUDA graphs (one per prefetch buffer set) and replayed."""
    import torch.distributed as dist

    result = {"ok": False}
    graphs, outs = [], []
    try:
        torch.cuda.synchronize()
        pool = None
        for b in range(2):
            batch = fetch.bufs[b]

            def step():
                pipe.invalidate_cache()
                pts_p.grad = None
                attrs_p.grad = None
                rgba, depth, _, _ = sharded.ShardedTraceRays.apply(tracer, pts_p, attrs_p, adj, off, batch["rays"],
                                                                   batch["start"], batch["dq"], False)
                loss = (((rgba - batch["target"]) ** 2).sum() / R_total
                        + 1e-4 * (depth[..., 0] - depth[..., 1]).abs().sum() / R_total)
                loss.backward()
                return loss.detach(), pts_p.grad, attrs_p.grad

            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(2):
                    step()
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, pool=pool):
                out = step()
            pool = g.pool()
            graphs.append(g)
            outs.append(out)
        ok = 1
    except Exception as e:  # noqa: BLE001
        result["error"] = repr(e)[:300]
        ok = 0
        try:
            torch.cuda.synchronize()
        except Exception:  # noqa: BLE001
            pass
    if world > 1:
        flag = torch.tensor([ok], dtype=torch.int32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        ok = int(flag.item())
    if not ok:
        result.setdefault("error", "capture failed on another rank")
        log(f"e2e CUDA graph unavailable: {result['error']}")
        return result

    def loop(steps, wall):
        nxt = fetch.enqueue(0)
        last = 0.0
        for i in range(steps):
            t0 = time.perf_counter()
            _, ev = nxt
            if i + 1 < steps:
                nxt = fetch.enqueue(i + 1)
            torch.cuda.current_stream(dev).wait_event(ev)
            graphs[i % 2].replay()
            last = float(outs[i % 2][0].item())  # D2H read of the step's result
            fetch.release(i)
            wall.append((time.perf_counter() - t0) * 1e3)
        return last

    loop(max(args.warmup, 3), [])
    gc.collect()
    gc.disable()
    barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    wall = []
    e0.record()
    loss = loop(args.steps, wall)
    e1.record()
    barrier(world)
    gc.enable()
    w = np.array(wall)
    result.update(ok=True, ms_per_step=max_over_ranks(e0.elapsed_time(e1), world) / args.steps, loss=loss,
                  wall_ms=[round(x, 2) for x in wall],
                  wall_stats={"min": float(w.min()), "median": float(np.median(w)), "max": float(w.max())})
    return result


def cpu_baseline(f, frame, log):
    """The CPU restatement (oracle/, OpenMP over the host cores) on a bounded sample of the
    same frame (8-row bands spread over it), sized for ~10-30 s.  Reported baseline, not a target."""
    from oracle import oracle

    H = frame["rays"].shape[0]
    # 8-row bands in a bit-reversal-like order (every 16th band first, then the bands between),
    # so that any prefix of the list is spread over the whole frame
    bands = sorted(range((H + 7) // 8), key=lambda b: (b % 16, b))
    rows = np.array([r for b in bands for r in range(8 * b, min(8 * b + 8, H))])
    cores = oracle.max_threads()

    def run(rsel):
        sl = {k: np.ascontiguousarray(v[np.sort(rsel)]) for k, v in frame.items()}
        t0 = time.time()
        fwd = oracle.trace_forward(f.points, f.attributes, f.adjacency, f.offsets, sl["rays"], sl["start"],
                                   sl["dq"], num_threads=0)
        oracle.trace_backward(f.points, f.attributes, f.adjacency, f.offsets, sl["rays"], sl["start"],
                              fwd["rgba"], sl["grad_rgba"], sl["dq"], fwd["depth_indices"], sl["grad_depth"],
                              num_threads=0)
        return time.time() - t0, sl["rays"].shape[0] * sl["rays"].shape[1]

    run(rows[:8])                       # spin the thread pool up
    t_probe, n_probe = run(rows[:64])   # ~6% of the frame
    want = int(min(len(rows), max(64, 64 * 15.0 / max(t_probe, 1e-3)))) // 8 * 8
    t, n = (t_probe, n_probe) if want <= 64 else run(rows[:want])
    log(f"cpu_baseline: {n} rays in {t:.1f} s on {cores} threads")
    return {"value": n / t / 1e6, "unit": "Mrays/s", "cores": cores, "kind": "port",
            "sample": f"{n} rays of the same frame ({want} of {H} rows, 8-row bands spread over the frame), "
                      f"fwd+bwd, C restatement of the path with OpenMP, {t:.1f} s; radfoam itself has no "
                      f"CPU tracing path"}


# ----------------------------------------------------------------------------- reference arm
def run_reference(args):
    """The reference's own CUDA kernels (src/tracing/pipeline.cu compiled unmodified into
    oracle/_ref) on ONE GPU, same workload, driven the way torch_bindings/pipeline_bindings.cpp
    and radfoam_model/render.py drive them (zero-filled grads, post-hoc finite scrub).  radfoam
    has no CPU tracing path and no multi-GPU path: under torchrun rank 0 alone runs."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch

    from oracle import ref_gpu

    log = lambda m: print(f"[bench-ref] {m}", file=sys.stderr, flush=True)  # noqa: E731
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    f = load_or_build_foam(args.points, log)
    frame = make_frame(f, args.width, args.height)
    H, W = args.height, args.width
    R = H * W
    if not ref_gpu.available():
        cpu = cpu_baseline(f, frame, log)
        print(json.dumps({"metric": METRIC, "value": cpu["value"], "unit": "Mrays/s", "n_gpus": 1,
                          "steps": 1, "warmup": 0, "ms_per_step": None, "higher_is_better": True,
                          "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                          "impl": "reference", "config": {"workload": "config4 sample on host cores "
                          "(oracle/_ref not built; CPU restatement)"}, "cpu_baseline": cpu,
                          "e2e": {"value": cpu["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0,
                                  "d2h_bytes_per_step": 0}}))
        return
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    points, attrs, adj, off = d(f.points), d(f.attributes), d(f.adjacency), d(f.offsets)
    host = {k: torch.from_numpy(v).pin_memory() for k, v in frame.items()}
    dv = {k: v.to(dev) for k, v in host.items()}

    def step_device():
        fwd = ref_gpu.trace_forward(points, attrs, adj, off, dv["rays"], dv["start"], dv["dq"])
        bwd = ref_gpu.trace_backward(points, attrs, adj, off, dv["rays"], dv["start"], fwd["rgba"],
                                     dv["grad_rgba"], dv["dq"], fwd["depth_indices"], dv["grad_depth"])
        pg, ag = bwd["points_grad"], bwd["attr_grad"]
        pg[~pg.isfinite()] = 0  # radfoam_model/render.py:98-99
        ag[~ag.isfinite()] = 0
        return fwd, bwd

    class RefTraceRays(torch.autograd.Function):  # radfoam_model/render.py:10-122 over oracle/_ref
        @staticmethod
        def forward(ctx, pts, at, rays, start, dq):
            res = ref_gpu.trace_forward(pts, at, adj, off, rays, start, dq)
            ctx.saved = (pts, at, rays, start, dq, res["rgba"], res["depth_indices"])
            return res["rgba"], res["depth"]

        @staticmethod
        def backward(ctx, g_rgba, g_depth):
            pts, at, rays, start, dq, rgba, didx = ctx.saved
            res = ref_gpu.trace_backward(pts, at, adj, off, rays, start, rgba, g_rgba.contiguous(), dq, didx,
                                         g_depth.contiguous())
            pg, ag = res["points_grad"], res["attr_grad"]
            pg[~pg.isfinite()] = 0
            ag[~ag.isfinite()] = 0
            return pg, ag, None, None, None

    pts_p, attrs_p = points.clone().requires_grad_(True), attrs.clone().requires_grad_(True)

    fetch = InputPrefetcher(host, ("rays", "start", "dq", "target"), dev)

    def step_e2e(batch, ev):
        torch.cuda.current_stream(dev).wait_event(ev)
        pts_p.grad = None
        attrs_p.grad = None
        rgba, depth = RefTraceRays.apply(pts_p, attrs_p, batch["rays"], batch["start"], batch["dq"])
        loss = (((rgba - batch["target"]) ** 2).sum() / R
                + 1e-4 * (depth[..., 0] - depth[..., 1]).abs().sum() / R)
        loss.backward()
        return loss

    def run_e2e(steps):
        nxt = fetch.enqueue(0)
        last = 0.0
        for i in range(steps):
            batch, ev = nxt
            if i + 1 < steps:
                nxt = fetch.enqueue(i + 1)
            last = float(step_e2e(batch, ev).item())
            fetch.release(i)
        return last

    for _ in range(max(args.warmup, 3)):
        fwd, _ = step_device()
    torch.cuda.synchronize()
    nint = fwd["num_intersections"].to(torch.int64)
    sampler = ClockSampler(0)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(args.steps):
        last_step = step_device()
    ev1.record()
    torch.cuda.synchronize()
    ms_per_step = ev0.elapsed_time(ev1) / args.steps
    dumped = (sample_outputs(dict(last_step[0], **last_step[1]), dv["rays"].shape[:-1], points.shape[0])
              if args.dump_outputs else None)
    del last_step
    clocks = sampler.stop()
    run_e2e(2)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    loss_val = run_e2e(args.steps)
    e1.record()
    torch.cuda.synchronize()
    e2e_ms = e0.elapsed_time(e1) / args.steps
    h2d = sum(host[k].numel() * host[k].element_size() for k in ("rays", "start", "dq", "target"))
    h2d_ms = fetch.last_copy_ms()
    value = R / (ms_per_step * 1e-3) / 1e6
    line = {
        "metric": METRIC, "value": value, "unit": "Mrays/s", "n_gpus": 1, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
        "config": {"workload": workload_name(f, W, H),
                   "step": "the reference's own CUDA kernels (prefetch_adjacent_diff + "
                           "forward/backward<float,3,128>, zero-fills, finite scrub) on one B200 -- radfoam ships "
                           "no CPU or multi-GPU tracing path",
                   "rays": R, "mean_cells_per_ray": float(nint.float().mean().item()),
                   "max_cells_per_ray": int(nint.max().item()), "parallelism": "single GPU"},
        "clocks": clocks,
        "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": 1, "kind": "reference",
                         "sample": "full frame; GPU kernels of the reference, one host launch thread"},
        "e2e": {"value": R / (e2e_ms * 1e-3) / 1e6, "unit": "Mrays/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 4, "loss": loss_val,
                "h2d_ms_per_step": h2d_ms, "h2d_overlapped": True},
    }
    if dumped is not None:
        dump_outputs(args.dump_outputs, dumped)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--points", type=int, default=1_048_576)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--emulate-shard", type=int, default=0,
                    help="single GPU only: trace rank 0's shard of an N-way ray split (profiling aid)")
    ap.add_argument("--kernel-times", action="store_true",
                    help="read per-kernel event timings inside the timed loop (serialises it)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's outputs (a fixed sample of rays and points) as DIR/<name>.npy; "
                         "with --gpus N > 1, rank 0's rays only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
    try:
        import torch.distributed as dist

        if dist.is_initialized():
            dist.destroy_process_group()
    except Exception:
        pass


if __name__ == "__main__":
    main()
