#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native reflect-sampling-nerf hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload train|render] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One "step" = one pass of the hot path over one batch of BASELINE.json configs[1]: 16,384 rays per GPU drawn from the
procedurally generated Blender-format shiny-sphere scene (100 views, 400x400; reflect_sampling_nerf_b200/data.py), 128
coarse + 128 fine samples, 64 + 64 reflected samples per bouncing ray, random-init field:
  train : pixel sampling + ray generation + get_outputs + get_loss_dict + backward + gradient all-reduce (N>1) + fused
          RAdam step + bf16 re-pack -- captured in one CUDA graph (N = 1)
  render: get_outputs in eval mode (BASELINE.json configs[2] chunk form)
Rays shard across ranks with no data-path collective (weak scaling: 16,384 rays per GPU); the only collective is the
per-step gradient all-reduce of the training workload.

Prints ONE JSON line (rank 0).  `value` = whole-job rays/s with the scene (cameras + uint8 images) resident in HBM;
`e2e` = the same through the public API (TrainStep.step(bundle, image): static-buffer copy + CUDA-graph replay at N = 1, eager at
N > 1) with HOST (pinned) ray / pixel buffers, H2D + D2H copies inside the timed region.  (The resident path generates its rays
on the GPU inside the step, the e2e path receives them from the host: the two differ by one small kernel vs 655 KB of H2D.)
`--impl reference` times the oracle restatement of the reference's PyTorch path on the host CPU cores
(the reference itself cannot be imported: nerfstudio is absent, SURVEY.md §8c).
`--dump-outputs DIR` writes what the timed path computed in its last timed step as DIR/<name>.npy (rank 0; see
step_outputs_to_host): the inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

import torch  # noqa: E402

CFG = dict(num_coarse_samples=128, num_importance_samples=128,
           num_reflect_coarse_samples=64, num_reflect_importance_samples=64)
RAYS_PER_GPU = 16384
SCENE = dict(n_views=100, resolution=400)     # BASELINE.json configs[1]: shiny sphere, 400x400, 100 views
FLOP_PRIMARY, FLOP_REFLECT, FLOP_INF = 1230592, 1229056, 1225472   # forward, per point (SURVEY.md §8d)
# dram__bytes_read.sum + dram__bytes_write.sum per work unit (point / sample), from ONE `ncu --set full` capture of each kernel
# at C2 primary-pass size (profiles/r02_field_all_v1_ncu.txt: 2,097,152 points; profiles/r02_composite16_*_ncu.txt: 65,536 x
# 128 samples).  `roofline.traffic` = this figure x the units the timed launches actually processed, per launch.
NCU_DRAM_BYTES_PER_UNIT = {
    "field_fwd_kernel": (0.010343e9 + 0.084744e9) / 2097152,
    "field_fwd_kernel[train]": (0.080746e9 + 10.652934e9) / 2097152,
    "field_chain_kernel<normals>": (1.075013e9 + 0.029699e9) / 2097152,
    "field_chain_kernel<backward>": (0.956941e9 + 9.354154e9) / 2097152,
    "field_wgrad_kernel": (20.880054e9 + 0.006595e9) / 2097152,
    "composite_fwd_kernel": (704.934656e6 + 37.376512e6) / (65536 * 128),
    "composite_bwd_kernel": (749.599744e6 + 522.126336e6) / (65536 * 128),
}


def scene_batch_cpu(n: int, seed: int, n_views: int = 8, resolution: int = 100):
    """A host-side batch of the same kind of rays (cameras on the radius-4 sphere, rays through the sphere scene) for the
    CPU / oracle arms: oracle/cameras.py ray arithmetic on a small in-memory instance of the scene."""
    from oracle import cameras as C
    from reflect_sampling_nerf_b200 import data as D
    cams = D.orbit_cameras(n_views, 4.0, resolution, resolution, 0.6911112070083618, seed=100)
    imgs = torch.stack([D.render_shiny_sphere(cams, i) for i in range(n_views)])
    g = torch.Generator().manual_seed(seed)
    pix = C.sample_pixels(torch.rand(n, 3, generator=g), n_views, resolution, resolution)
    o, d, area = C.generate_rays(cams.camera_to_worlds, cams.fx, cams.fy, cams.cx, cams.cy, pix)
    # pixel footprint of the 400x400 benchmark camera (the small instance only serves as a ray source)
    area = area * (resolution / SCENE["resolution"]) ** 2
    return o.contiguous(), d.contiguous(), area.contiguous(), C.gather_targets(imgs, pix)


class ClockSampler(threading.Thread):
    """SM clocks / throttle reasons DURING the timed region, through NVML in-process (no fork per sample)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag, self.err = index, [], threading.Event(), None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            try:
                self.power_limit_w = nv.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0
            except Exception:  # noqa: BLE001
                self.power_limit_w = None
            while not self.stop_flag.is_set():
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                try:
                    pw = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                except Exception:  # noqa: BLE001
                    pw = None
                self.samples.append((sm, mx, int(reasons), pw))
                self.stop_flag.wait(0.05)
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def summary(self):
        bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}
        sm = sorted(s[0] for s in self.samples)
        reasons = sorted({name for s in self.samples for name, b in bits.items() if s[2] & b})
        pw = sorted(s[3] for s in self.samples if s[3] is not None)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.samples[0][1] if self.samples else None,
                "reasons": reasons, "samples": len(self.samples), "power_w": pw[len(pw) // 2] if pw else None,
                "power_limit_w": getattr(self, "power_limit_w", None), "power_note": "NVML board power, ~1 s average", "source": "nvml", "error": self.err}


DUMP_RAYS, DUMP_SAMPLE_RAYS, DUMP_MAX_BYTES = 16384, 1024, 64 << 20


def step_outputs_to_host(outputs, loss=None, field=None):
    """What a caller of the timed path holds after its last step, copied to the host as float32 / float64 numpy arrays:
    the per-ray outputs of get_outputs, and for a training step the loss and the updated field parameters.  Per-ray
    outputs are those of a fixed, seeded sample of DUMP_RAYS rays (all of them for a batch no larger); per-sample outputs
    ([rays, samples, c]) those of the first DUMP_SAMPLE_RAYS rays of the sample.  `rays` = the sampled ray indices."""
    import numpy as np

    def host(t):
        t = t.detach().cpu()
        return t.numpy().astype(np.float64 if t.dtype in (torch.float64, torch.int64, torch.int32) else np.float32)

    n = next(iter(outputs.values())).shape[0]
    rays = torch.arange(n)
    if n > DUMP_RAYS:
        rays = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_RAYS].sort().values
    arrays = {"rays": rays.double().numpy()}
    for k, v in outputs.items():
        rows = rays[:DUMP_SAMPLE_RAYS] if v.dim() == 3 else rays
        arrays[k] = host(v[rows.to(v.device)])
    if loss is not None:
        arrays["loss"] = host(loss)
    if field is not None:
        arrays.update({"param." + k: host(p) for k, p in field.named_parameters()})
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes of outputs exceed {DUMP_MAX_BYTES}")
    return arrays


def dump_step_outputs(arrays, out_dir: str) -> None:
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


# ------------------------------------------------------------------------------------------ oracle arms
def oracle_step_rays_per_s(n_rays: int, workload: str, steps: int, warmup: int, device: str = "cpu",
                           autocast: bool = False, threads: int = 0):
    """The oracle restatement of the reference's PyTorch path (bounded sample of the workload) on `device`."""
    from oracle import upstream as U
    from oracle.refpath import OracleModel
    if threads:
        torch.set_num_threads(threads)
    torch.manual_seed(0)
    model = OracleModel(**CFG).to(device)
    model.train(workload == "train")
    opt = torch.optim.RAdam(model.field.parameters(), lr=1e-3, eps=1e-15)
    o, d, area, image = [t.to(device) for t in scene_batch_cpu(n_rays, 0)]
    times = []
    for i in range(warmup + steps):
        if device != "cpu":
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        bundle = U.RayBundle(origins=o, directions=d, pixel_area=area)
        with torch.autocast("cuda", dtype=torch.float16, enabled=autocast and device != "cpu"):
            if workload == "train":
                opt.zero_grad(set_to_none=True)
                out = model(bundle)
                loss = sum(model.get_loss_dict(out, {"image": image}).values())
                loss.backward()
                opt.step()
            else:
                with torch.no_grad():
                    model(bundle)
        if device != "cpu":
            torch.cuda.synchronize()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    sec = sum(times) / len(times)
    return n_rays / sec, sec


REF_SAMPLE_WHY = ("the full 16,384-ray step of the eager fp32 path holds ~60 GB of autograd activations and takes ~30 s per step "
                  "on the host cores; rays/s is size-normalised")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    n = args.ref_rays
    rps, sec = oracle_step_rays_per_s(n, args.workload, args.steps, args.warmup, threads=threads)
    line = {
        "impl": "reference", "metric": "rays_per_sec", "value": rps, "unit": "rays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"C2 {args.workload} step (128+128 samples, 64+64 reflected), bounded sample of "
                               f"{n} of {RAYS_PER_GPU} rays per step: {REF_SAMPLE_WHY}", "rays_per_step": n, **CFG},
        "cpu_baseline": {"value": rps, "unit": "rays/s", "cores": threads, "kind": "port",
                         "sample": f"{n} rays/step x {args.steps} steps, oracle restatement (PyTorch fp32 CPU); {REF_SAMPLE_WHY}"},
        "e2e": {"value": rps, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ B200 arm
def run_b200(args):
    import torch.distributed as dist
    from reflect_sampling_nerf_b200 import _lib, data, ops
    from reflect_sampling_nerf_b200.model import ReflectSamplingNeRFModel, ReflectSamplingNeRFModelConfig
    from reflect_sampling_nerf_b200.rays import RayBundle

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the rsn_b200 kernels have no CPU fallback")
    # NCCL prints its version banner on stdout at communicator creation: keep stdout clean for the ONE JSON line by
    # pointing fd 1 at stderr for the duration of the run and writing the result to the saved descriptor
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.call("rsn_device_ok")

    torch.manual_seed(1234 + rank)             # ranks start from DIFFERENT weights; TrainStep broadcasts rank 0's (as DDP does)
    model = ReflectSamplingNeRFModel(ReflectSamplingNeRFModelConfig(**CFG)).to(dev)
    train = args.workload == "train"
    model.train(train)
    n = args.rays
    # the scene: every rank renders the same 100 views and draws its own pixels (per-rank generator seed)
    cams, images = data.shiny_sphere_in_memory(SCENE["n_views"], SCENE["resolution"], device=dev)
    torch.cuda.manual_seed(1000 + rank)        # every rank draws its own pixels (default CUDA generator: graph-capturable)
    dm = data.RayDataManager(cams, images, rays_per_batch=n)
    # e2e: host-resident batches (pinned), the form the reference's CPU dataloader hands over
    with torch.no_grad():
        hb, hbatch = dm.next_train(0)
        host = [t.cpu().pin_memory() for t in (hb.origins, hb.directions, hb.pixel_area, hbatch["image"])]
    use_graph = train and args.graph in ("on", "auto")
    stepper = None
    if train:
        from reflect_sampling_nerf_b200.train_path import TrainStep
        stepper = TrainStep(model, world_size=world, lr_final=1e-4, max_steps=50000, graph=False)
    graph_stepper = None

    counters = {"launches": 0}
    orig_call = _lib.call

    def counting_call(name, *a):
        counters["launches"] += 1
        return orig_call(name, *a)
    _lib.call = counting_call
    ops._lib.call = counting_call

    loss_ring = {"i": 0, "ev": [None, None], "seen": [],
                 "buf": [torch.zeros((), dtype=torch.float32).pin_memory() for _ in range(2)]}

    def one_step(e2e: bool):
        if e2e and train:
            # the public API takes the pinned HOST batch as it is: TrainStep.step copies it to the device (into the static
            # input buffers of its CUDA graph once the step is captured) inside this timed call
            bundle = RayBundle(origins=host[0], directions=host[1], pixel_area=host[2])
            bi = host[3]
        elif e2e:
            bo, bd, ba, bi = [t.to(dev, non_blocking=True) for t in host]
            bundle = RayBundle(origins=bo, directions=bd, pixel_area=ba)
        else:
            bundle, batch = dm.next_train(0)           # pixel sampling + ray generation + target gather: one launch
            bi = batch["image"]
        if train:
            loss = stepper.step(bundle, bi)
            if e2e:
                # D2H read of the step's loss, consumed by the host one step late (pinned double buffer + event), the way
                # a training loop logs it: the copy is inside this step's timed region, the host never stalls the queue
                slot = loss_ring["i"] & 1
                if loss_ring["ev"][slot] is not None:
                    loss_ring["ev"][slot].synchronize()
                    loss_ring["seen"].append(float(loss_ring["buf"][slot]))
                loss_ring["buf"][slot].copy_(loss.detach().reshape(()), non_blocking=True)
                ev = torch.cuda.Event()
                ev.record()
                loss_ring["ev"][slot] = ev
                loss_ring["i"] += 1
            return loss
        out = model(bundle)
        if e2e:
            return out["mid_rgb_fine"].cpu(), out["mid_reflect_fine"].cpu()
        return out

    # CUDA-graph form of the resident-data training step: raygen + forward + losses + backward + optimizer in ONE graph
    graph_state = {}

    def build_graph():
        for _ in range(3):
            one_step(False)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        if world == 1:
            with torch.cuda.graph(g):
                bundle, batch = dm.next_train(0)
                graph_state["loss"] = stepper._eager(bundle, batch["image"])
            graph_state["replay"] = g.replay
            return g
        # N > 1: two graphs around the step's one collective (NCCL stays outside the captures), as TrainStep(graph=True)
        from reflect_sampling_nerf_b200.train_path import _allreduce_blob
        with torch.cuda.graph(g):
            bundle, batch = dm.next_train(0)
            graph_state["loss"] = stepper._forward_backward_tape(bundle, batch["image"], flush=False)
        blob = model.field._grad_blob
        g2 = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g2, pool=g.pool()):
            stepper.finish_step()

        def replay():
            g.replay()
            _allreduce_blob(model.field, blob)
            g2.replay()
        graph_state["replay"], graph_state["g2"] = replay, g2
        return g

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > L2 (126 MB)
    masked = []

    def timed(mode: str, steps: int, warmup: int):
        """mode: 'graph' (replay), 'eager' (resident data, PROFILE events on), 'e2e' (host buffers)."""
        e2e = mode == "e2e"
        run = graph_state["replay"] if mode == "graph" else (lambda: one_step(e2e))
        for _ in range(warmup):
            run()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ops.PROFILE = [] if mode == "eager" else None
        if mode in ("eager", "graph") and world > 1:
            model.field.__dict__["_allreduce_events"] = []
        counters["launches"] = 0
        evs, last = [], None
        for _ in range(steps):
            flush.zero_()                       # L2 flush between timed iterations (outside the event pairs)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            last = run()
            e1.record()
            evs.append((e0, e1))
            if mode != "e2e":
                masked.append(model.__dict__["last_num_bounced"].clone())     # device int32, read after the timed region
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        per_step = [a.elapsed_time(b) for a, b in evs]
        ms = sum(per_step)
        timed.last_per_step = per_step
        timed.last_result = graph_state["loss"] if mode == "graph" else last     # the loss (train) / outputs (render)
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        mine = t.clone()
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            allr = [torch.zeros_like(mine) for _ in range(world)]
            dist.all_gather(allr, mine)
            timed.per_rank = [float(x.item()) / steps for x in allr]
        else:
            timed.per_rank = [float(mine.item()) / steps]
        prof, ops.PROFILE = ops.PROFILE, None
        return float(t.item()) / steps, counters["launches"], prof

    sampler = ClockSampler(local) if rank == 0 else None
    cuda_graph = False
    if use_graph:
        try:
            graph_state["g"] = build_graph()
            cuda_graph = True
        except Exception as e:  # noqa: BLE001
            print(f"bench: CUDA graph capture failed ({e!r}); timing the eager step", file=sys.stderr)
            torch.cuda.synchronize()
    if sampler:
        sampler.start()
    ms_step, launches, _ = timed("graph" if cuda_graph else "eager", args.steps, args.warmup)
    step_ms = [round(x, 2) for x in timed.last_per_step]
    ar_main = model.field.__dict__.get("_allreduce_events") or []      # the timed steps' own all-reduce (N > 1)
    allreduce_ms_timed = (sum(a.elapsed_time(b) for a, b in ar_main) / len(ar_main)) if ar_main else None
    per_rank_ms = [round(x, 3) for x in timed.per_rank]
    if sampler:
        sampler.stop_flag.set()
        sampler.join(timeout=2)
    dumped = None
    if args.dump_outputs and rank == 0:
        # the last timed step's results, before the eager and e2e passes below train the model further
        dumped = (step_outputs_to_host(stepper.last_outputs, timed.last_result, model.field) if train
                  else step_outputs_to_host(timed.last_result))
    n_masked = [int(m) for m in masked] if masked else []
    # the same K steps eagerly, every instrumented kernel bracketed by CUDA events on the launching stream: the roofline's
    # launch durations (and the launch count of one step)
    masked.clear()
    if os.environ.get("RSN_BENCH_PROFILER_RANGE"):      # ncu --profile-from-start off: capture only the eager timed steps
        torch.cuda.profiler.start()
    ms_eager, launches_eager, prof = timed("eager", args.steps, 2)      # (2 warm-up steps: the first eager step after a graph replay re-binds workspaces)
    if os.environ.get("RSN_BENCH_PROFILER_RANGE"):
        torch.cuda.profiler.stop()
    ar_events = model.field.__dict__.pop("_allreduce_events", None) or []
    allreduce_ms = (sum(a.elapsed_time(b) for a, b in ar_events) / len(ar_events)) if ar_events else None
    if train and cuda_graph:
        # the public API's own CUDA-graph form (TrainStep(graph=True)): the host batch is copied into the graph's static
        # input buffers and the captured step is replayed -- the first step() below captures it
        stepper.graph_requested, stepper.steps_done = True, 3
    ms_e2e, _, _ = timed("e2e", args.steps, 3)

    # roofline: every field kernel from its own CUDA-event launch durations; `roofline` = the one with the largest
    # share of the step (tensor-bound kernels against the sustained cuBLAS bf16 peak, HBM-bound against the copy peak)
    roof, roof_all = None, []
    if prof:
        peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json"))) \
            if os.path.exists(os.path.join(REPO, "MEASURED_PEAKS.json")) else None
        tf_peak = peaks["bf16_tflops_sustained"] if peaks else 1400.0
        bw_peak = peaks["hbm_gbs"] if peaks else 6650.0
        src = "MEASURED_PEAKS.json (bf16_tflops_sustained: kernels timed inside a long step; hbm_gbs)" if peaks \
            else "B200_PROFILING.md fallback"
        by = {}
        for (name, a, b, flop, nbytes, count, cap_rays) in prof:
            # bounce passes: the launch is sized for the capacity, the work is what the device-side ray count covered
            scale = min(int(count), cap_rays) / cap_rays if (count is not None and cap_rays) else 1.0
            d = by.setdefault(name, [0.0, 0.0, 0.0, 0])
            d[0] += a.elapsed_time(b); d[1] += flop * scale; d[2] += nbytes * scale; d[3] += 1
        for name, (ms, flop, nbytes, cnt) in by.items():
            tf, gb = flop / ms / 1e9, nbytes / ms / 1e6
            hbm_bound = (gb / bw_peak) > (tf / tf_peak)
            roof_all.append({"kernel": name, "bound": "hbm" if hbm_bound else "tensor",
                             "achieved": gb if hbm_bound else tf, "peak": bw_peak if hbm_bound else tf_peak,
                             "unit": "GB/s" if hbm_bound else "TFLOP/s",
                             "frac": (gb / bw_peak) if hbm_bound else (tf / tf_peak),
                             "tflops": tf, "gbs": gb,
                             # measured DRAM bytes per launch: the per-unit figure of one ncu capture (NCU_DRAM_BYTES_PER_UNIT) x
                             # the units these launches processed; None for kernels without a capture
                             "traffic": (NCU_DRAM_BYTES_PER_UNIT[name] * (nbytes / ops.KERNEL_WORK[name][1]) / cnt
                                         if name in NCU_DRAM_BYTES_PER_UNIT else None),
                             "algorithmic_bytes": nbytes / cnt,
                             "launches": cnt, "avg_launch_ms": ms / cnt, "share_of_step": ms / (ms_eager * args.steps)})
        roof_all.sort(key=lambda r: -r["share_of_step"])
        roof = dict(roof_all[0], peak_source=src,
                    timed_in="an eager pass over the same K steps (the CUDA-graph replay cannot carry per-kernel events); "
                             "bounce-pass work is counted for the M rays the device-side count covered, not the launch capacity")

    cpu_base, cuda_base = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        rps, sec = oracle_step_rays_per_s(args.ref_rays, args.workload, 1, 1, threads=threads)
        cpu_base = {"value": rps, "unit": "rays/s", "cores": threads, "kind": "port",
                    "sample": f"{args.ref_rays} of {n} rays, 1 warm-up + 1 timed step ({sec:.1f} s), oracle restatement "
                              f"(PyTorch fp32 CPU) of the same {args.workload} step; {REF_SAMPLE_WHY}"}
    if rank == 0 and world == 1 and not args.no_cuda_baseline:
        # the north_star's >= 10x denominator: the reference-equivalent eager PyTorch path on THIS GPU, same step, same run
        del flush
        graph_state.clear()
        for key in ("_stash_pool", "_grad_blob_static", "_flat_grad"):
            model.field.__dict__.pop(key, None)
        model.field._dy_buffer = None
        torch.cuda.empty_cache()
        try:
            cuda_base = {"unit": "rays/s", "rays_per_step": n, "kind": "port (oracle restatement, eager PyTorch on cuda:0)"}
            for label, ac in (("fp32", False), ("fp16_autocast", True)):
                rps, sec = oracle_step_rays_per_s(n, args.workload, 2, 1, device=str(dev), autocast=ac)
                cuda_base[label] = rps
                cuda_base[label + "_ms_per_step"] = sec * 1e3
                torch.cuda.empty_cache()
        except Exception as e:  # noqa: BLE001
            cuda_base = {"error": repr(e)}

    if rank == 0:
        rays_total = n * world
        h2d = sum(t.numel() * t.element_size() for t in host)
        d2h = 4 if train else 2 * n * 3 * 4
        m_mean = sum(n_masked) / max(1, len(n_masked))
        s_p = CFG["num_coarse_samples"] + CFG["num_importance_samples"]
        s_r = CFG["num_reflect_coarse_samples"] + CFG["num_reflect_importance_samples"]
        samples_per_step = n * s_p + m_mean * (s_r + 1)              # SURVEY.md §8d: N (Sc+Sf) + M (Src+Srf) + M
        value = rays_total / (ms_step * 1e-3)
        line = {
            "metric": "rays_per_sec", "value": value, "unit": "rays/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"{args.config} {args.workload} step: {n} rays/GPU drawn on the GPU from the procedurally generated "
                                   f"Blender-format shiny-sphere scene ({SCENE['n_views']} views, {SCENE['resolution']}x"
                                   f"{SCENE['resolution']}) x (128 coarse + 128 fine) samples + reflected (64 + 64) per "
                                   f"bouncing ray, random-init field", "rays_per_gpu": n, **CFG,
                       "l2": "256 MB buffer written between timed iterations; per-pass field outputs (134 MB) exceed L2",
                       "parallelism": f"dp{world} (rays sharded, no data-path collective)",
                       "cuda_graph": (cuda_graph if world == 1 or not cuda_graph else
                                      "two graphs per step around the eager NCCL all-reduce of the gradient blob")},
            "field_samples_per_sec": samples_per_step * world / (ms_step * 1e-3),
            "masked_rays": {"mean_per_step_rank0": m_mean, "min": min(n_masked) if n_masked else None,
                            "max": max(n_masked) if n_masked else None, "of": n},
            "e2e": {"value": rays_total / (ms_e2e * 1e-3), "unit": "rays/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e,
                    "api": ("TrainStep.step(bundle, image) on pinned host buffers, CUDA-graph replay" if (train and cuda_graph)
                            else "TrainStep.step(bundle, image) on pinned host buffers, eager" if train
                            else "model(bundle) on pinned host buffers + D2H of the two rendered images")},
            "eager": {"ms_per_step": ms_eager, "gpu_launches_per_step": launches_eager / args.steps},
            "gpu_launches": launches if not cuda_graph else launches_eager,
            "gpu_launches_note": ("kernels launched by librsn_b200.so inside the timed region; with cuda_graph they are graph "
                                  "nodes replayed by one cudaGraphLaunch per step, counted from the eager pass of the same steps"),
            "step_ms_rank0": step_ms, "per_rank_step_ms": per_rank_ms, "allreduce_ms": allreduce_ms_timed if allreduce_ms_timed is not None else allreduce_ms,
            "clocks": sampler.summary() if sampler else None, "roofline": roof, "roofline_all": roof_all,
            "cpu_baseline": cpu_base, "cuda_baseline": cuda_base,
        }
        if cuda_base and "fp16_autocast" in cuda_base:
            line["vs_cuda_baseline"] = {"fp32": value / cuda_base["fp32"], "fp16_autocast": value / cuda_base["fp16_autocast"]}
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if dumped is not None:
        dump_step_outputs(dumped, args.dump_outputs)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="train", choices=["train", "render"])
    ap.add_argument("--rays", type=int, default=RAYS_PER_GPU)
    ap.add_argument("--config", default="C2", choices=["C2", "C3", "C5"],
                    help="BASELINE.json config: C2 = configs[1] train step, 16,384 rays per GPU (weak scaling; with --gpus 8 = "
                         "configs[3]); C3 = configs[2] render of one 800x800 frame, 640,000 rays sharded over the GPUs; C5 = "
                         "configs[4] render of 65,536 rays sharded over the GPUs (strong scaling)")
    ap.add_argument("--ref-rays", type=int, default=1024, help="bounded CPU sample (rays per oracle step)")
    ap.add_argument("--graph", default="auto", choices=["auto", "on", "off"],
                    help="CUDA-graph the training step (auto: single GPU only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cuda-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path computed in its last step as DIR/<name>.npy (float32 / float64, "
                         "at most 64 MB): per-ray outputs, and for training the loss and the updated field parameters; "
                         "with several GPUs, rank 0's rays only")
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    args.scaling = "weak"
    if args.config in ("C3", "C5"):
        args.workload, args.scaling = "render", "strong"
        total = 640000 if args.config == "C3" else 65536
        args.rays = (total + world - 1) // world
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs dumps the b200 path (--impl b200)")
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
