#!/usr/bin/env python
"""bench.py — augmented voxels/s of the 256^3 fp32 Compose pipeline on B200.

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA kernels)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path
    python bench.py ... --dump-outputs DIR                   # also save the last timed step's outputs

A "step" is one pass of the hot path over one batch of synthetic volumes:
``Compose([Affine, ElasticDeformation, BiasField, Blur, Noise, Gamma])`` on
``(B, 1, 256, 256, 256)`` fp32 (BASELINE.json configs[2]; ``--workload config2``
runs configs[1] = the first two transforms).  One process per GPU; every rank
augments its own batch (weak scaling, no data-path collective).

Prints ONE JSON line on rank 0 (keys documented in DESIGN.md §Measurement).
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
import warnings
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

VOL = 256
ALGO_BYTES_PER_VOXEL_RESAMPLE = 8  # one fp32 read + one fp32 write (SURVEY.md §8d)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="full", choices=["full", "config2"])
    ap.add_argument("--batch", type=int, default=32, help="volumes per GPU per step")
    ap.add_argument("--size", type=int, default=VOL)
    ap.add_argument("--noise", default=os.environ.get("TIO_B200_NOISE", "exact"),
                    choices=["exact", "philox"])
    ap.add_argument("--cpu-sample-batch", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-clocks", action="store_true", help="diagnostic: skip the nvidia-smi sampler")
    ap.add_argument("--no-numa", action="store_true", help="diagnostic: do not bind the rank to its GPU's NUMA node")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the configs[3] / configs[4] / gpu_baseline legs after the main timed region")
    ap.add_argument("--labels", action="store_true",
                    help="configs[3] shape: add an int16 LabelMap (nearest-neighbour resample) to every volume")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path,
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def pipeline_spec(workload):
    spec = [
        ("Affine", {"scales": (0.9, 1.1), "degrees": (-10, 10)}),
        ("ElasticDeformation", {}),
    ]
    if workload == "full":
        spec += [
            ("BiasField", {}),
            ("Blur", {"std": (0, 2)}),
            ("Noise", {"std": (0, 0.25)}),
            ("Gamma", {"log_gamma": (-0.3, 0.3)}),
        ]
    return spec


def synth_volumes(batch, size, pin):
    """(B,1,S,S,S) fp32 in [0,1): torch.rand(seed 1000+b) per element, on the host."""
    out = torch.empty((batch, 1, size, size, size), dtype=torch.float32, pin_memory=pin)
    for b in range(batch):
        g = torch.Generator().manual_seed(1000 + b)
        torch.rand((1, size, size, size), generator=g, out=out[b])
    return out


DUMP_BYTES = 32 << 20  # float32 voxel values written by --dump-outputs, over all images


def dump_outputs(batch, directory):
    """Write a step's outputs so that two builds can be compared output for output.

    Per image ``<name>`` of the batch: ``<name>_affines.npy``, the (B, 4, 4) float64 affines, and
    ``<name>.npy`` in float32: the whole (B, C, I, J, K) tensor when it fits DUMP_BYTES, else the
    voxels at flat indices ``torch.randint(numel, (n,), generator=torch.Generator().manual_seed(0))``,
    sorted, so that runs with the same arguments sample the same voxels."""
    import numpy as np

    directory.mkdir(parents=True, exist_ok=True)
    per_image = DUMP_BYTES // 4 // len(batch.images)
    for name, ib in batch.images.items():
        data = ib.data
        if data.numel() > per_image:
            g = torch.Generator().manual_seed(0)
            index = torch.randint(data.numel(), (per_image,), generator=g).sort().values
            data = data.reshape(-1)[index.to(data.device)]
        np.save(directory / f"{name}.npy", data.float().cpu().numpy())
        np.save(directory / f"{name}_affines.npy", np.stack([a.numpy() for a in ib.affines]).astype(np.float64))


# ----------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------


class ClockSampler:
    """nvidia-smi sampled every 200 ms during the timed region."""

    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-lms", "200", "-i", str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def wait_first_sample(self, timeout=10.0):
        """nvidia-smi takes a while to start: do not let its start-up overlap the timed region."""
        t0 = time.perf_counter()
        while self.proc is not None and not self.lines and time.perf_counter() - t0 < timeout:
            time.sleep(0.05)

    def stop(self, t_begin=None, t_end=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        window = [l for t, l in self.lines
                  if (t_begin is None or t >= t_begin) and (t_end is None or t <= t_end + 0.25)]
        if not window:  # region shorter than the sampling period: take the nearest samples
            window = [l for _, l in self.lines[-2:]]
        for line in window:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {
            "sm_mhz": sm[len(sm) // 2] if sm else None,
            "sm_max_mhz": max(smax) if smax else None,
            "reasons": sorted(reasons),
            "samples": len(sm),
        }


# ----------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------


def run_b200(args, rank, world, local_rank):
    import torch.distributed as dist

    import torchio_b200 as tio
    from torchio_b200 import ops

    from torchio_b200 import parallel

    os.environ["TIO_B200_NOISE"] = args.noise
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    # this rank's threads and (first-touch) pinned staging buffers next to its GPU
    numa = None if args.no_numa else parallel.bind_to_gpu_numa(local_rank)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        pipeline = tio.Compose(
            [getattr(tio, n)(**kw) for n, kw in pipeline_spec(args.workload)], copy=False)
    host = synth_volumes(args.batch, args.size, pin=True)
    resident = host.to(dev)
    affines = [tio.AffineMatrix() for _ in range(args.batch)]
    voxels = args.batch * args.size**3

    labels_host = labels_dev = None
    if args.labels:  # concentric boxes, values 0..4 (SURVEY.md §8d synthetic label)
        idx = torch.arange(args.size)
        ring = torch.minimum(idx, args.size - 1 - idx)
        depth = torch.minimum(torch.minimum(ring[:, None, None], ring[None, :, None]), ring[None, None, :])
        one = (depth * 5 // max(args.size // 2, 1)).clamp_(0, 4).to(torch.int16)
        labels_host = one[None, None].expand(args.batch, 1, -1, -1, -1).contiguous().pin_memory()
        labels_dev = labels_host.to(dev)

    def make_batch(tensor):
        images = {"t1": tio.ImagesBatch(tensor, list(affines))}
        if args.labels:
            images["seg"] = tio.ImagesBatch(labels_dev if tensor.is_cuda else labels_host, list(affines),
                                            image_class=tio.LabelMap)
        return tio.SubjectsBatch(images)

    # event hooks around the dominant kernel (K1) inside the real step
    k1_events = []
    raw_resample = ops.resample

    def timed_resample(*a, **kw):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        out = raw_resample(*a, **kw)
        e.record()
        k1_events.append((s, e))
        return out

    ops.resample = timed_resample

    def step(tensor):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            return pipeline(make_batch(tensor))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank) if (rank == 0 and not args.no_clocks) else None
    if sampler:
        sampler.start()
    torch.manual_seed(1234 + rank)
    for _ in range(args.warmup):
        out = step(resident)
    if sampler:
        sampler.wait_first_sample()
    k1_events.clear()
    barrier()
    launches0 = ops.launches()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    wall_begin = time.perf_counter()
    t0.record()
    for _ in range(args.steps):
        out = step(resident)
    t1.record()
    host_issue_ms = (time.perf_counter() - wall_begin) * 1e3 / args.steps
    barrier()
    wall_end = time.perf_counter()
    ms = t0.elapsed_time(t1)
    launches = ops.launches() - launches0
    clocks = sampler.stop(wall_begin, wall_end) if sampler else None
    k1_ms = [s.elapsed_time(e) for s, e in k1_events]
    if args.dump_outputs is not None and rank == 0:
        dump_outputs(out, args.dump_outputs)
    del out

    # end to end through the public call with HOST buffers: pinned input ->
    # H2D -> kernels -> D2H into pinned output, every step
    e2e = None
    if not args.no_e2e:
        def host_batches(n):
            for _ in range(n):
                yield make_batch(host)

        def run_stream(n, step_ms=None):
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                last, t_prev = None, time.perf_counter()
                for last in pipeline.stream(host_batches(n), depth=1):
                    if step_ms is not None:
                        now = time.perf_counter()
                        step_ms.append((now - t_prev) * 1e3)
                        t_prev = now
            return last

        def allocations():
            dev_stats = torch.cuda.memory_stats(dev)
            host_stats = torch.cuda.host_memory_stats() if hasattr(torch.cuda, "host_memory_stats") else {}
            return (dev_stats.get("num_device_alloc", 0), host_stats.get("num_host_alloc", 0))

        # (a) the loader-style public call: `for out in pipeline.stream(batches)` keeps one batch
        # in flight, so the copy-in of step n+1 overlaps the copy-out of step n; (b) the plain
        # call `pipeline(batch)`, step by step, reported beside it.
        # Warm-up: the loop keeps three pinned 2 GiB result buffers alive (in flight, yielded, held
        # by the consumer) and page-locking one takes ~0.6 s; device slices are cached by torch's
        # allocators too.  Warm up until a round of steps allocates nothing new.
        torch.manual_seed(4321 + rank)
        for _ in range(6):
            before = allocations()
            run_stream(max(4, args.warmup))
            if allocations() == before:
                break
        barrier()
        alloc0 = allocations()
        step_ms = []
        w0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = run_stream(args.steps, step_ms)
        e1.record()
        barrier()
        e2e_ms = max(e0.elapsed_time(e1), (time.perf_counter() - w0) * 1e3)
        alloc1 = allocations()
        assert res.images["t1"].data.device.type == "cpu"
        for _ in range(2):
            res = step(host)
        barrier()
        w0 = time.perf_counter()
        sync_steps = max(3, min(args.steps, 10))
        for _ in range(sync_steps):
            res = step(host)
        barrier()
        sync_ms = (time.perf_counter() - w0) * 1e3 / sync_steps
        moved = host.numel() * 4 + (labels_host.numel() * 2 if args.labels else 0)
        e2e = {"ms": e2e_ms, "bytes_in": moved, "bytes_out": moved, "sync_ms": sync_ms,
               "step_ms": [round(v, 1) for v in step_ms],
               "new_allocations": [alloc1[0] - alloc0[0], alloc1[1] - alloc0[1]]}
        del res
    ops.resample = raw_resample

    # the one exchange the north-star names: augmented volumes of every rank -> rank 0 (NCCL
    # send/recv over NVLink), timed on its own and reported beside the augmentation throughput
    gather = None
    if world > 1:
        out = step(resident)
        counts = [args.batch] * world
        dest = parallel.gather_buffers(out, counts) if rank == 0 else None
        for _ in range(2):
            parallel.gather_batch_to_root(out, counts=counts, out=dest)
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        reps = max(3, min(args.steps, 10))
        for _ in range(reps):
            parallel.gather_batch_to_root(out, counts=counts, out=dest)
        g1.record()
        barrier()
        gather = {"ms": g0.elapsed_time(g1) / reps,
                  "bytes_into_root": (world - 1) * sum(ib.data.numel() * ib.data.element_size()
                                                       for ib in out.images.values())}
        del out, dest

    extras = {}
    if rank == 0 and not args.no_extras and world == 1:
        extras = extra_legs(args, dev, pipeline_spec, tio, ops)

    if world > 1:
        t = torch.tensor([ms, e2e["ms"] if e2e else 0.0, gather["ms"]], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t[0])
        if e2e:
            e2e["ms"] = float(t[1])
        gather["ms"] = float(t[2])
    if rank != 0:
        return None

    peaks = {}
    peaks_path = ROOT / "MEASURED_PEAKS.json"
    if peaks_path.exists():
        peaks = json.loads(peaks_path.read_text())
    peak = float(peaks.get("hbm_gbs", 6650.0))
    k1_avg_ms = sum(k1_ms) / len(k1_ms) if k1_ms else float("nan")
    achieved = ALGO_BYTES_PER_VOXEL_RESAMPLE * voxels / (k1_avg_ms * 1e-3) / 1e9
    value = world * voxels * args.steps / (ms * 1e-3)
    line = {
        "metric": "augmented voxels/sec on 256^3 fp32 Compose pipeline",
        "value": value,
        "unit": "voxels/s",
        "n_gpus": world,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": ms / args.steps,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f32",
        "data": "synthetic",
        "config": {
            "workload": ("configs[2]: batch %d of 1x%d^3 fp32, Compose(Affine, ElasticDeformation,"
                         " BiasField, Blur, Noise, Gamma) per GPU" % (args.batch, args.size))
            + (" + int16 LabelMap (nearest)" if args.labels else "")
            if args.workload == "full" else
            ("configs[1]: batch %d of 1x%d^3 fp32, Compose(Affine, ElasticDeformation) per GPU"
             % (args.batch, args.size)),
            "global_batch": world * args.batch,
            "parallelism": f"dp{world} (independent volumes, no data-path collective)",
            "noise_normals": args.noise,
            "l2_policy": "inputs (%.1f GiB/GPU) larger than L2 (126 MB)" % (voxels * 4 / 2**30),
            "includes": "host param sampling + table upload + all kernels of the step",
        },
        "gpu_launches": launches,
        "host_issue_ms_per_step": host_issue_ms,
        "roofline": {
            "kernel": "K1 = tile_bounds_kernel + resample_fast_kernel (%d launches in the timed region)" % len(k1_ms),
            "bound": "hbm",
            "achieved": achieved,
            "peak": peak,
            "unit": "GB/s",
            "frac": achieved / peak,
            "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s",
            "algorithmic_bytes_per_launch": ALGO_BYTES_PER_VOXEL_RESAMPLE * voxels,
            "avg_launch_ms": k1_avg_ms,
            "share_of_step": sum(k1_ms) / ms if k1_ms else None,
            "traffic": k1_traffic(args),
            "traffic_source": "profiles/r2_k1_traffic.json (committed ncu --set full capture, not this run)",
        },
        "clocks": clocks,
    }
    if e2e:
        line["e2e"] = {
            "value": world * voxels * args.steps / (e2e["ms"] * 1e-3),
            "unit": "voxels/s",
            "h2d_bytes_per_step": e2e["bytes_in"],
            "d2h_bytes_per_step": e2e["bytes_out"],
            "ms_per_step": e2e["ms"] / args.steps,
            "api": "for out in pipeline.stream(host_batches, depth=1): one batch in flight, every batch copied"
                   " in from pinned host memory and its result copied back inside the timed region",
            "plain_call_ms_per_step": e2e["sync_ms"],
            "step_ms": e2e["step_ms"],
            "new_device_host_allocations_in_timed_region": e2e["new_allocations"],
        }
    if numa is not None:
        line["config"]["numa"] = numa
    if gather:
        gbs = gather["bytes_into_root"] / (gather["ms"] * 1e-3) / 1e9
        step_ms = ms / args.steps
        line["gather"] = {
            "what": "parallel.gather_batch_to_root: every rank's augmented batch -> rank 0, NCCL send/recv",
            "ms": gather["ms"],
            "bytes_into_root": gather["bytes_into_root"],
            "gb_per_s": gbs,
            "frac_of_900_gbs_root_ingest": gbs / 900.0,
            "value_with_gather": world * voxels / ((step_ms + gather["ms"]) * 1e-3),
            "value_without_gather": value,
        }
    line.update(extras)
    if not args.no_cpu_baseline and world == 1:
        line["cpu_baseline"] = cpu_reference(args, steps=3, warmup=1)
    return line


def extra_legs(args, dev, pipeline_spec, tio, ops):
    """Measured after the main region (N = 1): configs[3]'s per-GPU shape (image + int16 label
    map), configs[4]'s patch path, and the reference's op sequence on CUDA tensors."""
    out = {}
    size, batch = args.size, args.batch
    voxels = batch * size**3
    # ---- configs[3]: batch of fp32 image + int16 LabelMap, full Compose ----
    if args.workload == "full" and not args.labels:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            pipe = tio.Compose([getattr(tio, n)(**kw) for n, kw in pipeline_spec("full")], copy=False)
        idx = torch.arange(size)
        ring = torch.minimum(idx, size - 1 - idx)
        depth = torch.minimum(torch.minimum(ring[:, None, None], ring[None, :, None]), ring[None, None, :])
        one = (depth * 5 // max(size // 2, 1)).clamp_(0, 4).to(torch.int16)
        labels = one[None, None].expand(batch, 1, -1, -1, -1).contiguous().to(dev)
        images = torch.rand((batch, 1, size, size, size), device=dev)
        affines = [tio.AffineMatrix() for _ in range(batch)]
        label_ms = []
        raw = ops.resample

        def timed(src, *a, **kw):
            if src.dtype != torch.int16:
                return raw(src, *a, **kw)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            r = raw(src, *a, **kw)
            e.record()
            label_ms.append((s, e))
            return r

        ops.resample = timed

        def one_step():
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                return pipe(tio.SubjectsBatch({
                    "t1": tio.ImagesBatch(images, list(affines)),
                    "seg": tio.ImagesBatch(labels, list(affines), image_class=tio.LabelMap)}))

        torch.manual_seed(77)
        for _ in range(3):
            one_step()
        label_ms.clear()
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        steps = 5
        t0.record()
        for _ in range(steps):
            one_step()
        t1.record()
        torch.cuda.synchronize()
        ops.resample = raw
        ms = t0.elapsed_time(t1) / steps
        lab = [s.elapsed_time(e) for s, e in label_ms]
        lab_avg = sum(lab) / len(lab)
        peak = 6576.4
        peaks_path = ROOT / "MEASURED_PEAKS.json"
        if peaks_path.exists():
            peak = float(json.loads(peaks_path.read_text()).get("hbm_gbs", peak))
        out["config3"] = {
            "workload": "configs[3] per-GPU shape: batch %d of (1x%d^3 fp32 image + int16 LabelMap, nearest),"
                        " full Compose, resident" % (batch, size),
            "ms_per_step": ms,
            "value": voxels / (ms * 1e-3),
            "unit": "voxels/s",
            "label_pass": {
                "kernel": "resample_tile_kernel<int16, nearest> (%d launches)" % len(lab),
                "avg_launch_ms": lab_avg,
                "algorithmic_bytes_per_voxel": 4,
                "achieved_gb_s": 4 * voxels / (lab_avg * 1e-3) / 1e9,
                "frac_of_hbm_peak": 4 * voxels / (lab_avg * 1e-3) / 1e9 / peak,
            },
        }
        del labels, images
        torch.cuda.empty_cache()
    # ---- configs[4]: Queue(128^3 patches, 8 per volume, max_length 512) -> dummy 3-D UNet forward ----
    try:
        out["config4"] = queue_unet_leg(args, dev, tio)
    except Exception as exc:  # never lose the headline line to an extra
        out["config4"] = {"error": repr(exc)}
    # ---- the reference's op sequence on CUDA tensors (the existing Blackwell path) ----
    if not args.no_cpu_baseline:
        try:
            out["gpu_baseline"] = gpu_reference(args, dev)
        except Exception as exc:
            out["gpu_baseline"] = {"error": repr(exc)}
    return out


def queue_unet_leg(args, dev, tio):
    """configs[4] on one GPU: subjects of 1x256^3 -> Compose on the device -> 8 patches of 128^3 per
    volume into the device patch ring (max_length 512 would be 4 GiB; 64 here) -> batches of 8 ->
    forward of a small conv3d encoder/decoder.  patches/s, augmentation + extraction + forward."""
    import torch.nn as nn

    size = args.size
    n_subjects, per_volume, patch, batch_size, max_length = 16, 8, 128, 8, 64
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        pipe = tio.Compose([getattr(tio, n)(**kw) for n, kw in pipeline_spec("full")], copy=False)
    subjects = []
    for i in range(n_subjects):
        g = torch.Generator().manual_seed(2000 + i)
        subjects.append(tio.Subject(t1=tio.ScalarImage(torch.rand((1, size, size, size), generator=g))))
    sampler = tio.UniformSampler(subjects[0], patch)
    queue = tio.Queue(subjects, max_length=max_length, patches_per_volume=per_volume, patch_sampler=sampler,
                      transform=pipe, num_workers=0, shuffle_subjects=False, shuffle_patches=True, device=dev)
    loader = tio.SubjectsLoader(queue, batch_size=batch_size)
    net = nn.Sequential(
        nn.Conv3d(1, 8, 3, padding=1), nn.ReLU(inplace=True), nn.Conv3d(8, 16, 3, stride=2, padding=1),
        nn.ReLU(inplace=True), nn.Conv3d(16, 16, 3, padding=1), nn.ReLU(inplace=True),
        nn.ConvTranspose3d(16, 8, 2, stride=2), nn.ReLU(inplace=True), nn.Conv3d(8, 2, 1),
    ).to(dev).to(memory_format=torch.channels_last_3d).half()
    torch.manual_seed(5)
    with torch.no_grad(), warnings.catch_warnings():  # warm-up: cuDNN plan, kernels, the ring itself
        warnings.simplefilter("ignore")
        for batch in tio.SubjectsLoader(tio.Queue(subjects[:2], max_length=max_length, patches_per_volume=per_volume,
                                                  patch_sampler=sampler, transform=pipe, shuffle_subjects=False,
                                                  device=dev), batch_size=batch_size):
            net(batch.images["t1"].data.half().contiguous(memory_format=torch.channels_last_3d))
    n_patches = 0
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    with torch.no_grad(), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for batch in loader:
            x = batch.images["t1"].data
            y = net(x.half().contiguous(memory_format=torch.channels_last_3d))
            n_patches += x.shape[0]
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    assert y.shape[0] > 0
    return {
        "workload": "configs[4] on one GPU: Queue(%d subjects of 1x%d^3 on the host, Compose of six on the device,"
                    " UniformSampler(%d), patches_per_volume=%d, max_length=%d, device ring) ->"
                    " SubjectsLoader(batch_size=%d) -> conv3d encoder/decoder forward (fp16)"
                    % (n_subjects, size, patch, per_volume, max_length, batch_size),
        "patches": n_patches,
        "seconds": dt,
        "value": n_patches / dt,
        "unit": "patches/s",
        "patch_voxels_per_s": n_patches * patch**3 / dt,
        "includes": "H2D of each subject, augmentation, patch gather, UNet forward",
    }


def gpu_reference(args, dev):
    """The reference's op sequence (oracle/torch_port.py = what TorchIO runs) on CUDA tensors of
    the same B200: the existing Blackwell path the fused kernels are compared with."""
    import numpy as np

    import torchio_b200 as tio
    from oracle import torch_port

    b, size = 2, args.size
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        transforms = [getattr(tio, n)(**kw) for n, kw in pipeline_spec(args.workload)]
    data = synth_volumes(b, size, pin=False)
    batch = tio.SubjectsBatch({"t1": tio.ImagesBatch(data, [tio.AffineMatrix() for _ in range(b)])})
    resident = data.to(dev)

    def one_step():
        history = []
        for t in transforms:
            torch.rand(1)
            history.append({"name": type(t).__name__, "params": t.make_params(batch)})
        images = {"t1": {"kind": "scalar", "data": resident, "affines": [np.eye(4) for _ in range(b)]}}
        with warnings.catch_warnings(), torch.device(dev):
            warnings.simplefilter("ignore")
            torch_port.replay(images, history)
        return images["t1"]["data"]

    torch.manual_seed(99)
    one_step()
    torch.cuda.synchronize()
    times = []
    for _ in range(3):
        t0 = time.perf_counter()
        one_step()
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    times.sort()
    torch.cuda.empty_cache()
    return {
        "value": b * size**3 / times[1],
        "unit": "voxels/s",
        "kind": "port-on-cuda",
        "sample": f"median of 3 steps of batch {b} x 1x{size}^3 fp32, same Compose, torch {torch.__version__}"
                  " CUDA ops (ATen sm_100 kernels) on the same GPU, inputs resident, host randn + H2D as the reference does",
        "seconds_per_step": times[1],
        "spread_s": [times[0], times[-1]],
    }


# ----------------------------------------------------------------------------
# reference arm / CPU baseline: the oracle's torch-op port = the op sequence
# the reference executes on the host (oracle/torch_port.py)
# ----------------------------------------------------------------------------


def k1_traffic(args):
    """DRAM bytes per K1 launch (dram__bytes_read.sum + dram__bytes_write.sum, mean of the affine and
    the elastic launch) from the committed `ncu --set full` capture of this workload
    (profiles/r2_k1_traffic.json) — not re-measured in this run — or None when the run differs."""
    path = ROOT / "profiles" / "r2_k1_traffic.json"
    if not path.exists() or args.batch != 32 or args.size != VOL:
        return None
    return json.loads(path.read_text()).get("bytes_per_launch")


def cpu_reference(args, steps, warmup):
    import numpy as np

    import torchio_b200 as tio
    from oracle import torch_port

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    # bounded sample: ~13 s per step at batch 2 on the GPU box's 128 host threads; one volume per
    # step for long runs keeps the whole --steps run within a few minutes
    b = args.cpu_sample_batch if steps * args.cpu_sample_batch <= 12 else 1
    size = args.size
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        transforms = [getattr(tio, n)(**kw) for n, kw in pipeline_spec(args.workload)]
    data = synth_volumes(b, size, pin=False)
    batch = tio.SubjectsBatch(
        {"t1": tio.ImagesBatch(data, [tio.AffineMatrix() for _ in range(b)])})

    def one_step():
        # sample params with the product's host code (identical to the
        # reference's sampling, tests/test_host_params.py), replay on CPU ops
        history = []
        for t in transforms:
            torch.rand(1)
            history.append({"name": type(t).__name__, "params": t.make_params(batch)})
        images = {"t1": {"kind": "scalar", "data": data,
                         "affines": [np.eye(4) for _ in range(b)]}}
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            torch_port.replay(images, history)

    torch.manual_seed(99)
    for _ in range(max(warmup, 1)):
        one_step()
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        one_step()
        times.append(time.perf_counter() - t0)
    dt = sum(times)
    ordered = sorted(times)
    median = ordered[len(ordered) // 2]
    return {
        "value": b * size**3 / median,
        "unit": "voxels/s",
        "cores": cores,
        "kind": "port",
        "sample": f"median of {steps} step(s) (after {max(warmup, 1)} warm-up) of batch {b} x 1x{size}^3 fp32, "
                  f"same Compose, torch {torch.__version__} CPU ops, {torch.get_num_threads()} threads",
        "seconds": dt,
        "batch": b,
        "median_step_s": median,
        "spread_step_s": [ordered[0], ordered[-1]],
        "warmup": max(warmup, 1),
    }


def run_reference(args, rank, world):
    if rank != 0:
        return None
    base = cpu_reference(args, steps=args.steps, warmup=min(args.warmup, 1))
    return {
        "impl": "reference",
        "metric": "augmented voxels/sec on 256^3 fp32 Compose pipeline",
        "value": base["value"],
        "unit": "voxels/s",
        "n_gpus": world,
        "steps": args.steps,
        "warmup": base["warmup"],
        "ms_per_step": base["median_step_s"] * 1e3,
        "step_spread_ms": [x * 1e3 for x in base["spread_step_s"]],
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f32",
        "data": "synthetic",
        "config": {
            "workload": "bounded sample of the same Compose: batch %d of 1x%d^3 per step on the"
                        " host cores (rank 0 only); value = voxels per MEDIAN step" % (base["batch"], args.size),
            "parallelism": "host threads",
        },
        "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": base["value"], "unit": "voxels/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        line = run_reference(args, rank, world)
        if line is not None:
            print(json.dumps(line), flush=True)
        return
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        line = run_b200(args, rank, world, local_rank)
        if line is not None:
            print(json.dumps(line), flush=True)
    finally:
        if world > 1:
            import torch.distributed as dist

            dist.destroy_process_group()


if __name__ == "__main__":
    main()
