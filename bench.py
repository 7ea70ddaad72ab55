#!/usr/bin/env python
"""bench.py -- rays/s (fwd+bwd) of the volumetric render hot path on BASELINE.json's config 2.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--res 1024] [--scene lego|dense] [--dump-outputs DIR]

One "step" = one pass of the hot path over one 1024x1024 frame of synthetic rays:
    Pipeline(NeuralRadianceField(HashGrid L=16,F=2,T=2^19; decoders 32-64-16 / 42-64-64-3), PackedRFTracer('ray', 2048))
    forward -> huber loss vs a synthetic target image -> backward -> (N>1: NCCL all-reduce of the gradients) -> fused Adam step.
`value`  : whole-job rays/s with rays and target already resident in HBM.
`e2e`    : the same step driven from HOST buffers: rays + target copied H2D from pinned memory and the loss read back
           D2H inside the timed region, through the public Pipeline call.
`--impl reference`: the CPU restatement of the reference path (oracle, OpenMP, all host cores) on a bounded ray sample.
Rank 0 prints ONE JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "rays/sec (fwd+bwd) 1024^2 Lego NeRF HashGrid"
CAM_ORIGIN, CAM_LOOKAT, CAM_FOV, NEAR, FAR = [-3.0, 0.65, -3.0], [0.0, 0.0, 0.0], 30.0, 0.0, 10.0   # nerf_hash.yaml:111-118


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--res", type=int, default=1024)
    ap.add_argument("--num-steps", type=int, default=2048)
    ap.add_argument("--scene", default="lego", choices=["lego", "dense"])
    ap.add_argument("--trace-host", action="store_true", help="print host-side phase times of every step to stderr (diagnostics)")
    ap.add_argument("--premarch", type=int, default=1, help="1: march batch i+1 on a side stream while batch i renders (PackedRFTracer.premarch)")
    ap.add_argument("--precision", type=int, default=1, help="0: fp32 decoders, 1: fp16 tensor-core decoders (reference enable_amp)")
    ap.add_argument("--cpu-sample-rays", type=int, default=0, help="rays in the CPU-baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--step-api", default="native", choices=["native", "autograd"],
                    help="native: wisp_b200.MultiviewStep (the trainer step as one native sequence: fused loss, one-launch Adam); "
                         "autograd: Pipeline call + torch loss + loss.backward() + torch fused Adam (the round-1 step)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N > 1: weak = N views per step (1024^2 rays per GPU, the default the driver runs); strong = ONE view per step tiled over "
                         "the N GPUs (rows rank::N each), SURVEY 8(e) inference-style partitioning")
    ap.add_argument("--config", type=int, default=2, choices=[1, 2, 3, 4],
                    help="BASELINE.json config: 1 = HashGrid 8-level, 1-layer-32 MLP, 256^2 single view (the reference's CPU-runnable case; same runner as 2), "
                         "2 = HashGrid NeRF fwd+bwd (headline), 3 = nglod OctreeGrid SDF sphere trace, 4 = TriplanarGrid NeRF")
    ap.add_argument("--hidden-dim", type=int, default=0, help="configs 1/2: decoder width override (128 = the reference's best published app/nerf setting)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (its outputs and the parameters it updated) as DIR/<name>.npy, "
                         f"float32 or float64, at most {DUMP_LIMIT // 10**6} MB in all, to compare two builds on the same inputs")
    a = ap.parse_args()
    if a.config == 1 and a.res == 1024:
        a.res = 256
    return a


def metric_name(args):
    return METRIC if args.config != 1 else "rays/sec (fwd+bwd) 256^2 single-view NeRF HashGrid 8-level (BASELINE configs[0])"


def nef_shape(args):
    """(num_lods, hidden_dim) of the benched field: configs[1] (headline) unless --config 1 (configs[0])."""
    L, H = (8, 32) if args.config == 1 else (16, 64)
    return L, (args.hidden_dim or H)


def make_onef(O, args):
    L, H = nef_shape(args)
    return O.make_nef(feature_std=1e-4, seed=0, num_lods=L, hidden_dim=H)


def workload_config(args):
    L, H = nef_shape(args)
    return {"workload": f"app/nerf HashGrid {L}-level F=2 T=2^19, {'2-layer-64' if H == 64 else f'num_layers=1 hidden-{H}'} MLP, {args.res}^2 rays x {args.num_steps} steps ('ray'), "
                        f"{'lego-like level-7 octree' if args.scene == 'lego' else 'dense level-7 octree'}, fwd+bwd+Adam",
            "rays_per_step_per_gpu": args.res * args.res // (args.gpus if getattr(args, "scaling", "weak") == "strong" else 1), "num_steps": args.num_steps, "scene": args.scene,
            "camera": {"origin": CAM_ORIGIN, "lookat": CAM_LOOKAT, "fov": CAM_FOV, "near": NEAR, "far": FAR},
            "loss": "huber/rays", "optimizer": ("Adam on table + decoders: one native launch (wb_adam_step)" if args.step_api == "native"
                                                else "Adam(fused, torch) on table + decoders"),
            "step_api": ("wisp_b200.MultiviewStep.step (mirror of MultiviewTrainer.step: no autograd, loss fused into the compositing backward)"
                         if args.step_api == "native" else "Pipeline(rays) -> torch smooth_l1_loss -> loss.backward() -> torch.optim.Adam(fused)"),
            "pipeline": ("march of batch i+1 enqueued on a side stream while batch i renders (one march per timed step, none carried "
                         "in from the warm-up)") if args.premarch else "none",
            "l2": "per-step working set (hit masks + sample records, >1 GB) exceeds the 126 MB L2; a different camera every step",
            "parallelism": (f"dp{args.gpus}: {args.gpus} views per step, every rank renders rows rank::{args.gpus} of each view (same sample load on "
                            f"every rank), NCCL all-reduce of gradients") if args.gpus > 1 else "single GPU"}


DUMP_LIMIT = 64_000_000          # bytes of array data written by --dump-outputs


def dump_outputs(path, arrays, limit=DUMP_LIMIT):
    """Write each array as <path>/<name>.npy, float64 where it was computed so and float32 otherwise.  The limit is shared out from
    the smallest array up; an array larger than its share is replaced by a fixed, seeded sample of its rows, and the indices of
    those rows are written beside it as <name>.rows.npy."""
    os.makedirs(path, exist_ok=True)
    arrays = {k: np.asarray(v) for k, v in arrays.items()}
    arrays = {k: np.ascontiguousarray(v, dtype=np.float64 if v.dtype == np.float64 else np.float32) for k, v in arrays.items()}
    left = limit
    for i, (name, a) in enumerate(sorted(arrays.items(), key=lambda kv: (kv[1].nbytes, kv[0]))):
        share = left // (len(arrays) - i)
        if a.nbytes > share:
            row_bytes = a.nbytes // a.shape[0]
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], share // (row_bytes + 8), replace=False))
            np.save(os.path.join(path, name + ".rows.npy"), rows.astype(np.float64))
            a = a[rows]
            left -= rows.size * 8
        np.save(os.path.join(path, name + ".npy"), a)
        left -= a.nbytes


def host_arrays(named):
    """name -> host copy of each tensor, float64 kept, everything else as float32 (bool masks become 0 / 1)."""
    import torch
    return {k: (v.detach() if v.dtype == torch.float64 else v.detach().float()).cpu().numpy() for k, v in named.items()}


def orbit_origin(i: int):
    """Camera i of the orbit: the reference camera rotated about the y axis."""
    a = 2.0 * np.pi * (i % 360) / 360.0 * 7.0
    x, z = CAM_ORIGIN[0], CAM_ORIGIN[2]
    return [float(x * np.cos(a) - z * np.sin(a)), CAM_ORIGIN[1], float(x * np.sin(a) + z * np.cos(a))]


# ------------------------------------------------------------------------------------------------------------------
# CPU arm (oracle): cpu_baseline of the GPU line and the whole `--impl reference` run
# ------------------------------------------------------------------------------------------------------------------
def cpu_scene(args):
    from oracle import oracle as O
    onef = make_onef(O, args)                                         # config 2 shapes (config 1 with --config 1)
    pts = O.lego_like_points(7)
    spc = O.octree_to_spc(O.points_to_octree(pts, 7) if args.scene == "lego" else O.dense_octree(7))
    return O, onef, spc


def cpu_time_step(O, onef, spc, args, nrays, cam_i, seed, keep=None):
    """One bounded sample: `nrays` rays strided uniformly over the res^2 frame of camera cam_i, full config."""
    o, d = O.look_at_rays(orbit_origin(cam_i), CAM_LOOKAT, args.res, args.res, CAM_FOV)
    R = o.shape[0]
    sel = (np.arange(nrays, dtype=np.int64) * R) // nrays
    o, d = np.ascontiguousarray(o[sel]), np.ascontiguousarray(d[sel])
    tgt = (1.0 / (1.0 + np.exp(-np.random.default_rng(2).standard_normal((nrays, 3))))).astype(np.float32)
    t0 = time.perf_counter()
    st = O.rf_step(spc, onef, o, d, NEAR, FAR, args.num_steps, tgt, loss="huber", bg=(0, 0, 0), seed=seed)
    dt = time.perf_counter() - t0
    if keep is not None:                      # parity leg of the GPU arm: the oracle's outputs and the inputs that produced them
        keep.update(st=st, origins=o, dirs=d, target=tgt, seed=seed)
    return dt, st["num_samples"]


def use_all_host_threads(O):
    """The CPU arm always runs on every host core: torchrun exports OMP_NUM_THREADS=1 to its workers, which would silently
    turn the OpenMP oracle into a single-thread run (round-1 SCALE ratios at N >= 2 were void for that reason)."""
    n = os.cpu_count() or 1
    try:
        n = max(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    O.set_num_threads(n)
    return O.num_threads()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    O, onef, spc = cpu_scene(args)
    cores = use_all_host_threads(O)
    nrays = args.cpu_sample_rays or 65536
    for i in range(args.warmup):              # warm-up at the timed size (page-faults of the 42 MB gradient table, thread pool spin-up)
        cpu_time_step(O, onef, spc, args, nrays, i, i)
    times, samples, last = [], 0, {}
    for i in range(args.steps):
        dt, ns = cpu_time_step(O, onef, spc, args, nrays, args.warmup + i, args.warmup + i, keep=last)
        times.append(dt); samples += ns
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last["st"])
    med = float(np.median(times))             # median of the steps: robust against a noisy neighbour on the shared host
    value = nrays / med
    sample = (f"{nrays} rays strided over the {args.res}^2 frame per step, full config (n={args.num_steps}); "
              f"{samples // max(args.steps, 1)} hit samples/step; value = rays / median step time")
    line = {"impl": "reference", "metric": metric_name(args), "value": value, "unit": "rays/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * med, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(args),
            "cpu_baseline": {"value": value, "unit": "rays/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "step_s": [round(t, 4) for t in times],
            "note": "reference has no CPU tracer and cannot be built here (kaolin un-vendored); this is the oracle port, OpenMP on all host cores"}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 200 ms (the interval of the profiling recipe) while the timed regions run."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        if os.environ.get("WB_BENCH_NO_SAMPLER"):      # diagnostics: is a stall caused by the nvidia-smi poll?
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index), "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
            # nvidia-smi's start-up (driver enumeration, seconds on a fresh box) stalls kernel launches of this process for tens of ms:
            # wait for its first row here, outside every timed region (seen as a 14 ms "step" in a 1.5 ms-per-step configuration)
            t0 = time.perf_counter()
            while not self.rows and time.perf_counter() - t0 < 8.0 and self.proc.poll() is None:
                time.sleep(0.02)
            self.idle_rows = len(self.rows)
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass
        if len(self.rows) > getattr(self, "idle_rows", 0):       # rows read before the warm-up started describe an idle GPU
            self.rows = self.rows[self.idle_rows:]
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[j] for r in self.rows if len(r) >= 7 for j in range(4) if r[3 + j].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


def run_ours(args):
    import torch
    import torch.distributed as dist
    import wisp_b200 as W
    from oracle import oracle as O           # scene description + CPU baseline only; never on the measured GPU path

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus or world == 1, (world, args.gpus)

    # ---- model: identical init on every rank, taken from the oracle's seeded numpy init so that the CPU restatement and the GPU
    # model are the SAME network (the parity leg below compares them on the cpu_baseline sample) ----
    torch.manual_seed(0)
    onef0 = make_onef(O, args)                                        # config 2 shapes; pure numpy (no oracle library call)
    n_lods, hidden = nef_shape(args)
    pts = torch.from_numpy(O.lego_like_points(7))
    blas = W.OctreeAS.from_quantized_points(pts.to(dev), 7) if args.scene == "lego" else W.OctreeAS.make_dense(7, device=dev)
    grid = W.HashGrid.from_geometric(blas, feature_dim=2, num_lods=n_lods, multiscale_type='cat', feature_std=1e-4, codebook_bitwidth=19,
                                     min_grid_res=16, max_grid_res=512)
    nef = W.NeuralRadianceField(grid, view_embedder='positional', view_multires=4, hidden_dim=hidden, num_layers=1, bias=True).to(dev)
    with torch.no_grad():
        grid.codebook.feats.copy_(torch.from_numpy(onef0.table))
        for dec, Ws, bs in ((nef.decoder_density, onef0.dens_W, onef0.dens_b), (nef.decoder_color, onef0.col_W, onef0.col_b)):
            for l, Wm, bm in zip(list(dec.layers) + [dec.lout], Ws, bs):
                l.weight.copy_(torch.from_numpy(np.ascontiguousarray(Wm))); l.bias.copy_(torch.from_numpy(np.ascontiguousarray(bm)))
    tracer = W.PackedRFTracer(raymarch_type='ray', num_steps=args.num_steps, bg_color=(0.0, 0.0, 0.0))
    tracer.precision = args.precision
    pipe = W.Pipeline(nef, tracer)
    params = [p for p in nef.parameters() if p.requires_grad]
    native = args.step_api == "native"
    if native:        # the trainer step as one native sequence (flattens the decoder parameters in place)
        stepper = W.MultiviewStep(pipe, lr=1e-3, eps=1e-15, rgb_loss_type="huber", rgb_loss_denom="rays", precision=args.precision)
    else:
        opt = torch.optim.Adam(params, lr=1e-3, eps=1e-15, fused=True)
        reducer = W.parallel.GradientReducer(params)

    R = args.res * args.res
    nsteps_total = args.warmup + args.steps
    # ---- inputs: `world` cameras per step; rank k takes image rows k::world of each of them (R rays per rank: weak scaling with the
    # same occupancy statistics on every rank, instead of one whole view per rank whose sample count differs by camera);
    # host copies pinned for the e2e leg ----
    host_rays, host_tgt = [], []
    g = torch.Generator().manual_seed(2)
    for i in range(nsteps_total):
        os_, ds_ = [], []
        for c in range(world if args.scaling == "weak" else 1):
            o, d = O.look_at_rays(orbit_origin(i * world + c if args.scaling == "weak" else i), CAM_LOOKAT, args.res, args.res, CAM_FOV)
            o, d = o.reshape(args.res, args.res, 3)[rank::world], d.reshape(args.res, args.res, 3)[rank::world]
            os_.append(o.reshape(-1, 3)); ds_.append(d.reshape(-1, 3))
        o, d = np.ascontiguousarray(np.concatenate(os_)), np.ascontiguousarray(np.concatenate(ds_))
        host_rays.append((torch.from_numpy(o).pin_memory(), torch.from_numpy(d).pin_memory()))
        host_tgt.append(torch.sigmoid(torch.randn(o.shape[0], 3, generator=g)).pin_memory())
    R = host_rays[0][0].shape[0]
    dev_rays = [(o.to(dev), d.to(dev)) for o, d in host_rays]
    dev_tgt = [t.to(dev) for t in host_tgt]

    def seed_of(i):
        return 1000 + i * world + rank

    host_trace = []                        # --trace-host: wall-clock of the host-side phases of every step (diagnostics only)
    last_rgb = [None]                      # --dump-outputs, autograd step: the image of the latest step

    def step(i, origins, dirs, target, nxt=None, nxt_ready=None):
        import time
        t0 = time.perf_counter()
        if native:
            # software pipeline of the training loop: the sample selection of batch i+1 (it depends on rays + occupancy, not on the
            # weights) is enqueued on a side stream before batch i is rendered.  Every timed step enqueues exactly one march.
            nr = W.Rays(nxt[0], nxt[1], dist_min=NEAR, dist_max=FAR) if (nxt is not None and args.premarch) else None
            loss = stepper.step(W.Rays(origins, dirs, dist_min=NEAR, dist_max=FAR), target, seed=seed_of(i), next_rays=nr, next_seed=seed_of(i + 1),
                                next_ready=nxt_ready)
            if args.trace_host:
                host_trace.append((i, round((time.perf_counter() - t0) * 1e3, 2), torch.cuda.memory_stats(dev).get("num_device_alloc", 0)))
            return loss
        if nxt is not None and args.premarch:
            tracer.premarch(nef, W.Rays(nxt[0], nxt[1], dist_min=NEAR, dist_max=FAR), seed_of(i + 1), ready=nxt_ready)
        t1 = time.perf_counter()
        opt.zero_grad(set_to_none=True)      # autograd then adopts the returned gradient buffers: no zero-fill + accumulate pass over the 42 MB table
        tracer.seed = seed_of(i)
        rb = pipe(rays=W.Rays(origins, dirs, dist_min=NEAR, dist_max=FAR), lod_idx=None, channels=["rgb"])
        if args.dump_outputs:
            last_rgb[0] = rb.rgb.detach()
        t2 = time.perf_counter()
        loss = torch.nn.functional.smooth_l1_loss(rb.rgb, target, reduction='none').mean()       # multiview_trainer.py:144-154
        t3 = time.perf_counter()
        loss.backward()
        t4 = time.perf_counter()
        reducer.reduce()                      # N>1: NCCL all-reduce(mean) of table + decoder gradients; no-op at N=1
        opt.step()
        if args.trace_host:
            t5 = time.perf_counter()
            host_trace.append((i, round((t1 - t0) * 1e3, 2), round((t2 - t1) * 1e3, 2), round((t3 - t2) * 1e3, 2), round((t4 - t3) * 1e3, 2),
                               round((t5 - t4) * 1e3, 2), torch.cuda.memory_stats(dev).get("num_device_alloc", 0)))
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- parity at bench scale, on the benched path: the GPU step vs the CPU restatement on the cpu_baseline sample (same rays,
    # same jitter seed, same weights, full config) BEFORE any training step; also times the CPU run -> cpu_baseline ----
    parity, cpu_base = None, None
    if rank == 0 and not args.no_cpu_baseline:
        parity, cpu_base = parity_leg(args, O, W, torch, dev, spc_np=None, onef=onef0, pipe=pipe, tracer=tracer, nef=nef, stepper=stepper if native else None)
    W.ops.reserve_samples(int(1.08 * 16.0e6 * (args.res / 1024.0) ** 2 * (args.num_steps / 2048.0)) if args.scene == "lego" else 0)
    sampler = ClockSampler(local)          # started before the warm-up so that samples exist for short timed regions; it keeps
    if rank == 0:                          # running (one nvidia-smi process, 200 ms period) through both timed loops
        sampler.start()
    # ---- warm-up ----
    # The warm-up exercises the same pipeline, but nothing is carried over into the timed region.  Its LAST step marches its own batch
    # on the main stream (no pre-marched batch is left for it), exactly as the first timed step will: torch's caching allocator keeps
    # one pool per stream, and a first timed step that is the only one to march on the main stream after the pool has been carved up by
    # the other warm-up steps would pay a cudaMalloc inside the timed region (seen as one 37 ms step of 17.8 and
    # cudaMalloc_calls_in_timed_region = 1).
    for i in range(args.warmup):
        step(i, *dev_rays[i], dev_tgt[i], nxt=dev_rays[i + 1] if i + 1 < args.warmup - 1 else None)
    barrier()

    # ---- timed: device-resident inputs ----
    W.ops.PROFILE = []
    launches0 = W._cabi.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    dev_allocs0 = torch.cuda.memory_stats(dev).get("num_device_alloc", 0)
    step_ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    e0.record()
    step_ev[0].record()
    total_samples = 0
    for k in range(args.steps):
        i = args.warmup + k
        loss = step(i, *dev_rays[i], dev_tgt[i], nxt=dev_rays[i + 1] if k + 1 < args.steps else None)
        total_samples += tracer.get_prev_num_samples()
        step_ev[k + 1].record()
    e1.record()
    barrier()
    dumped = None
    if args.dump_outputs and rank == 0:   # before the e2e leg below takes further optimiser steps
        dumped = host_arrays({"loss": loss, "rgb": stepper.last_rgb if native else last_rgb[0], **dict(nef.named_parameters())})
    ms = e0.elapsed_time(e1)
    step_ms = [step_ev[k].elapsed_time(step_ev[k + 1]) for k in range(args.steps)]
    dev_allocs = torch.cuda.memory_stats(dev).get("num_device_alloc", 0) - dev_allocs0
    launches = W._cabi.launch_count() - launches0
    prof = W.ops.PROFILE
    W.ops.PROFILE = None
    stage_ms = {}
    for name, a, b in prof:
        stage_ms.setdefault(name, []).append(a.elapsed_time(b))

    # ---- timed: end to end from host buffers through the public API ----
    copy_stream = torch.cuda.Stream(device=dev)

    def e2e_pass(first, count, timed_events=None):
        batches = [(host_rays[first + k][0], host_rays[first + k][1], host_tgt[first + k]) for k in range(count)]
        pre = W.parallel.HostPrefetcher(batches, dev, stream=copy_stream)
        last = None
        for k, (o, d, t) in enumerate(pre):                    # every step's H2D copy and march are inside the pass
            loss = step(first + k, o, d, t, nxt=pre.staged, nxt_ready=pre.staged_event)
            last = float(loss.item())                          # device -> host read of the step's result
            if timed_events is not None:
                timed_events[k + 1].record()
        return last

    e2e_pass(0, args.warmup)                                   # untimed: warms the copy stream's allocator pool and the pipeline
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2e_ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    e2.record(); e2e_ev[0].record()
    loss_host = e2e_pass(args.warmup, args.steps, e2e_ev)
    e3.record()
    barrier()
    e2e_step_ms = [e2e_ev[k].elapsed_time(e2e_ev[k + 1]) for k in range(args.steps)]
    ms_e2e = e2.elapsed_time(e3)

    # ---- extra (SURVEY.md 8(d) "also forward-only rays/s"): inference render of the same frames, no gradients ----
    render = None
    try:
        with torch.no_grad():
            n_r = min(3, args.steps)
            r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            pipe(rays=W.Rays(*dev_rays[0], dist_min=NEAR, dist_max=FAR), lod_idx=None, channels=["rgb"])      # untimed
            torch.cuda.synchronize()
            r0.record()
            for k in range(n_r):
                tracer.seed = seed_of(args.warmup + k)
                pipe(rays=W.Rays(*dev_rays[args.warmup + k], dist_min=NEAR, dist_max=FAR), lod_idx=None, channels=["rgb"])
            r1.record()
            torch.cuda.synchronize()
            render = {"value": R * n_r / (r0.elapsed_time(r1) * 1e-3), "unit": "rays/s", "ms_per_frame": r0.elapsed_time(r1) / n_r,
                      "what": "forward only (march + shade + composite), device-resident rays, per GPU"}
    except Exception as ex:                                    # never let the extra figure break the contract line
        render = {"error": repr(ex)[:200]}
    clocks = sampler.stop() if rank == 0 else None

    per_rank = None
    if world > 1:       # where the step time goes on every rank (SURVEY 8(e)): samples, step time, stage times incl. the gradient all-reduce
        mine = {"rank": rank, "samples_per_step": total_samples / max(args.steps, 1), "ms_per_step": ms / max(args.steps, 1),
                "stage_ms": {k: round(float(np.mean(v)), 4) for k, v in stage_ms.items()}}
        per_rank = [None] * world
        dist.all_gather_object(per_rank, mine)
    tms = torch.tensor([ms, ms_e2e, float(total_samples), float((render or {}).get("ms_per_frame", float("nan")))], dtype=torch.float64, device=dev)
    if world > 1:
        mx = tms.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = tms.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        ms, ms_e2e, total_samples = float(mx[0]), float(mx[1]), float(sm[2])
        if render and "ms_per_frame" in render:        # forward-only at N GPUs: every rank renders its share concurrently, max over ranks
            render.update(ms_per_frame=float(mx[3]), value=R * world / (float(mx[3]) * 1e-3),
                          what=f"forward only (march + shade + composite), device-resident rays, aggregate over {world} GPUs, max over ranks (unsynchronised start)")
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    rays_total = R * args.steps * world          # R = rays per rank per step (weak: res^2, strong: res^2 / world)
    value = rays_total / (ms * 1e-3)
    e2e_value = rays_total / (ms_e2e * 1e-3)
    S_step = total_samples / (args.steps * world)

    # ---- rooflines (SURVEY.md 8(d): algorithmic bytes per hit sample; DESIGN.md section 4) ----
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    tfl = float(peaks.get("bf16_tflops_sustained", 1400.0))            # kernels timed inside a long step -> sustained figure
    src = "MEASURED_PEAKS.json (measured)" if peaks else "fallback 6650 GB/s / 1400 TFLOP/s"
    traffic = {}
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))     # dram bytes per launch from the last ncu --set full capture
    except Exception:
        pass
    e = 4                                                      # fp32 table and fp32 gradients
    L_eff = n_lods - 1                                         # 'cat' zeroes the last LOD (hash_grid.py:228): 15 of 16 levels are live
    dec_flop = 2 * (2 * n_lods * hidden + hidden * 16 + (15 + 27) * hidden + hidden * hidden + hidden * 3)   # one forward pass of both decoders (20096 at config 2)
    mean_ms = {k: float(np.mean(v)) for k, v in stage_ms.items()}
    models = {   # stage -> (kernel, bound, algorithmic units per hit sample, unit)
        "shade_fwd": ("wb_shade_fwd_tc_kernel" if args.precision == 1 else "wb_shade_fwd_kernel", "hbm", L_eff * 8 * 2 * e, "B"),
        "table_scatter": ("wb_table_scatter_kernel", "hbm", 2 * L_eff * 8 * 2 * e, "B"),
        # the fused backward kernel moves, per hit sample, the 64 B of saved features in and the read-modify-write of the table entries
        # (2 * L * 8 * F * 4 B): that is its SURVEY 8(d) figure; its decoder FLOPs are reported as a second line below
        "shade_bwd": (((("wb_mlp_bwd3_tc_kernel<FUSE> (decoder backward + table scatter)" if hidden in (64, 128) else "wb_mlp_bwd_tc_kernel + wb_table_scatter_kernel (one stage)"),
                        "hbm", 4 * n_lods + 2 * L_eff * 8 * 2 * e, "B")) if args.precision == 1
                      else ("wb_shade_bwd_kernel", "hbm", 2 * L_eff * 8 * 2 * e, "B")),
        "decoder_bwd": ("wb_mlp_bwd_tc_kernel", "tensor", 3 * dec_flop, "FLOP"),     # forward recompute + data grad + weight grad of both decoders
    }
    rooflines = []
    for st_name, (kern, bound, per, unit) in models.items():
        if st_name not in mean_ms:
            continue
        t_s = mean_ms[st_name] * 1e-3
        if bound == "hbm":
            ach, peak, u = S_step * per / t_s / 1e9, hbm, "GB/s"
        else:
            ach, peak, u = S_step * per / t_s / 1e12, tfl, "TFLOP/s"
        tr = traffic.get(kern)
        rooflines.append({"bound": bound, "kernel": kern, "achieved": ach, "peak": peak, "unit": u, "frac": ach / peak,
                          "traffic": tr, "kernel_ms": mean_ms[st_name], "algorithmic_per_sample": f"{per} {unit}", "samples_per_launch": S_step})
        kshort = kern.split("<")[0].split(" ")[0]
        if traffic.get(kshort + "__l2_pct") is not None:       # the table is L2-resident: where the launch sits against the L2 roof (ncu, same command)
            rooflines[-1]["l2_frac"] = traffic[kshort + "__l2_pct"] / 100.0
            rooflines[-1]["l2_source"] = f"ncu lts__throughput.avg.pct_of_peak_sustained_elapsed, profiles/{traffic.get('tag', '')}_{kshort}.txt"
            if tr is None:
                rooflines[-1]["traffic"] = traffic.get(kshort)
        if bound == "hbm":
            rooflines[-1]["note"] = "algorithmic table bytes; the table is L2-resident, so this is HBM-equivalent and can exceed 1 (see `traffic`)"
    if args.precision == 1 and "shade_bwd" in mean_ms:   # the same launch against the tensor roof: recompute + data grad + weight grad of both decoders
        t_s = mean_ms["shade_bwd"] * 1e-3
        ach = S_step * (3 * dec_flop) / t_s / 1e12
        rooflines.append({"bound": "tensor", "kernel": "wb_mlp_bwd3_tc_kernel<FUSE> (decoder part)", "achieved": ach, "peak": tfl, "unit": "TFLOP/s", "frac": ach / tfl,
                          "traffic": traffic.get("wb_mlp_bwd3_tc_kernel"), "kernel_ms": mean_ms["shade_bwd"] - 1e-9, "algorithmic_per_sample": f"{3 * dec_flop} FLOP",
                          "samples_per_launch": S_step, "note": "same launch as the hbm line of this kernel; the decoder rounds alone take 3.7 of its 7.0 ms (profiles/README.md)"})
    roofline = dict(max(rooflines, key=lambda r: r["kernel_ms"]))
    roofline["peak_source"] = src
    roofline["note"] = ("dominant kernel by time.  hbm-bound kernels: the 41.7 MB table is L2 resident, so `achieved` is HBM-equivalent gather/scatter "
                        "bandwidth and DRAM `traffic` is far below the algorithmic bytes (no wasted re-reads); see DESIGN.md section 4")

    line = {"metric": metric_name(args), "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f32" if args.precision == 0 else "f16(tensor)+f32 accumulate", "data": "synthetic", "config": workload_config(args),
            "e2e": {"value": e2e_value, "unit": "rays/s", "h2d_bytes_per_step": R * (24 + 12), "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps,
                    "step_ms": e2e_step_ms, "last_loss": loss_host},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "rooflines": rooflines,
            "march": {"candidates_per_step": R * args.num_steps, "candidates_per_sec": R * args.num_steps / (mean_ms.get("march_count", float("nan")) * 1e-3)},
            "samples_per_step_per_gpu": S_step, "samples_per_sec": total_samples / (ms * 1e-3), "stage_ms": mean_ms,
            "step_ms": step_ms, "cudaMalloc_calls_in_timed_region": int(dev_allocs), "render_only": render, "per_rank": per_rank}

    if cpu_base is not None:
        line["cpu_baseline"] = cpu_base
        line["parity"] = parity
    if args.trace_host:
        print("step, premarch ms, zero_grad+forward ms, loss ms, backward ms, reduce+opt ms, cudaMallocs so far", file=sys.stderr)
        for row in host_trace:
            print(row, file=sys.stderr)
    if dumped is not None:
        dump_outputs(args.dump_outputs, dumped)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()



# ------------------------------------------------------------------------------------------------------------------
# parity at bench scale (rank 0, outside every timed region)
# ------------------------------------------------------------------------------------------------------------------
PARITY_TOL = {0: {"rgb": 1e-4, "loss": 1e-5, "grad": 2e-3}, 1: {"rgb": 2e-3, "loss": 2e-3, "grad": 3e-2}}    # DESIGN.md "Tolerances"


def parity_leg(args, O, W, torch, dev, spc_np, onef, pipe, tracer, nef, stepper=None):
    """The CPU restatement and the GPU pipeline on the same bounded sample of the benched frame: per-ray rgb, the huber loss and the
    gradients of one step.  Raises if a tolerance is exceeded: a fast step whose result differs from the reference's is not a result."""
    use_all_host_threads(O)
    spc = O.octree_to_spc(O.points_to_octree(O.lego_like_points(7), 7) if args.scene == "lego" else O.dense_octree(7))
    R = args.res * args.res
    dt0, _ = cpu_time_step(O, onef, spc, args, 2048, 0, 0)                          # probe, then size the sample to ~12 s of CPU work
    nr = args.cpu_sample_rays or int(min(R, max(4096, 2048 * 12.0 / max(dt0, 1e-3))))
    keep = {}
    dt, ns = cpu_time_step(O, onef, spc, args, nr, args.warmup, 1000 + args.warmup, keep=keep)
    cpu_base = {"value": nr / dt, "unit": "rays/s", "cores": O.num_threads(), "kind": "port",
                "sample": f"{nr} rays strided over the {args.res}^2 frame, full config, {ns} hit samples, {dt:.1f} s"}
    st = keep["st"]
    for p_ in nef.parameters():
        p_.grad = None
    tracer.seed = keep["seed"]
    o, d, tgt = (torch.from_numpy(keep[k]).to(dev) for k in ("origins", "dirs", "target"))
    if stepper is not None:       # the benched step itself (MultiviewStep): its loss, its rgb and its gradient buffers, before they are cleared
        loss = stepper.step(W.Rays(o, d, dist_min=NEAR, dist_max=FAR), tgt, seed=keep["seed"], zero_grad=False, local_only=True, update=False)
        torch.cuda.synchronize()
        rgb_gpu = stepper.last_rgb.cpu().numpy()
        g_table, g_dens, g_col = stepper.g_grid[0].cpu().numpy(), stepper.g_dens.cpu().numpy(), stepper.g_col.cpu().numpy()
        stepper.zero_grads()
    else:
        rb = pipe(rays=W.Rays(o, d, dist_min=NEAR, dist_max=FAR), lod_idx=None, channels=["rgb"])
        loss = torch.nn.functional.smooth_l1_loss(rb.rgb, tgt, reduction='none').mean()
        loss.backward()
        torch.cuda.synchronize()
        flat = lambda dec: torch.cat([t.grad.reshape(-1) for l in list(dec.layers) + [dec.lout] for t in (l.weight, l.bias)]).cpu().numpy()
        rgb_gpu = rb.rgb.detach().cpu().numpy()
        g_table, g_dens, g_col = nef.grid.codebook.feats.grad.cpu().numpy(), flat(nef.decoder_density), flat(nef.decoder_color)

    def rel(a, b):
        return float(np.abs(a - b).max() / max(float(np.abs(b).max()), 1e-30))
    out = {"rays": int(nr), "samples": int(ns), "samples_match": bool(tracer.get_prev_num_samples() == st["num_samples"]),
           "precision": int(args.precision),
           "step_api": "native" if stepper is not None else "autograd",
           "rgb_max_abs_err": float(np.abs(rgb_gpu - st["rgb"]).max()),
           "loss_gpu": float(loss.detach()), "loss_cpu": float(st["loss"]), "loss_rel_err": abs(float(loss.detach()) - st["loss"]) / max(abs(st["loss"]), 1e-30),
           "table_grad_rel_err": rel(g_table, st["table"]),
           "density_decoder_grad_rel_err": rel(g_dens, st["dens"]),
           "color_decoder_grad_rel_err": rel(g_col, st["col"]),
           "tolerance": PARITY_TOL[int(args.precision)], "checked_against": "oracle/wisp_oracle.c wo_rf_step (fp32), same rays / seed / weights"}
    tol = out["tolerance"]
    ok = (out["samples_match"] and out["rgb_max_abs_err"] <= tol["rgb"] and out["loss_rel_err"] <= tol["loss"]
          and max(out["table_grad_rel_err"], out["density_decoder_grad_rel_err"], out["color_decoder_grad_rel_err"]) <= tol["grad"])
    out["ok"] = bool(ok)
    for p_ in nef.parameters():
        p_.grad = None
    if not ok:
        print(json.dumps({"parity_failure": out}), file=sys.stderr, flush=True)
        raise SystemExit("bench.py: GPU result differs from the CPU restatement beyond the stated tolerance (see stderr)")
    return out, cpu_base


# ------------------------------------------------------------------------------------------------------------------
# BASELINE config 3 (app/nglod OctreeGrid SDF sphere trace) and config 4 (TriplanarGrid NeRF): single GPU per rank
# ------------------------------------------------------------------------------------------------------------------
def _peaks():
    try:
        pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(pk.get("hbm_gbs", 6650.0)), "MEASURED_PEAKS.json (measured)"
    except Exception:
        return 6650.0, "fallback 6650 GB/s (B200_PROFILING.md)"


def _ncu_facts(roof: dict, key: str) -> dict:
    """DRAM bytes per launch and L2 utilisation of kernel `key` from the last ncu capture of the same command (profiles/traffic.json)."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        return roof
    if t.get(key) is not None:
        roof["traffic"] = t[key]
    if t.get(key + "__l2_pct") is not None:
        roof["l2_frac"] = t[key + "__l2_pct"] / 100.0
        roof["l2_source"] = f"ncu lts__throughput.avg.pct_of_peak_sustained_elapsed, profiles/{t.get('tag', '')}_{key}.txt"
    return roof


def _finish_line(args, torch, dist, world, rank, dev, line_fn, ms, ms_e2e, extra):
    tms = torch.tensor([ms, ms_e2e] + list(extra), dtype=torch.float64, device=dev)
    if world > 1:
        mx = tms.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = tms.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        tms = torch.cat([mx[:2], sm[2:]])
    if rank == 0:
        print(json.dumps(line_fn(float(tms[0]), float(tms[1]), [float(x) for x in tms[2:]])), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_config3(args):
    """One step = one 512^2 frame through Pipeline(NeuralSDF(OctreeGrid F=16, 6 LODs, 'sum', 128-wide decoder), PackedSDFTracer(32, 0.8)):
    native raytrace + ONE persistent sphere-tracing kernel (wb_sdf_trace) + finite-difference normals (nglod_octree.yaml)."""
    import torch
    import torch.distributed as dist
    import wisp_b200 as W
    from oracle import octree_grid as OG
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from gpu_util import sdf_nef_from_case
    world, rank, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local); dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    res = 512 if args.res == 1024 else args.res
    nsteps, step_size, min_dis = 32, 0.8, 3e-4
    case = OG.make_sdf_case(level=7, num_lods=6, feature_dim=16, hidden_dim=128, multiscale="sum", res=64, seed=11, feature_std=0.02)
    nef = sdf_nef_from_case(case, device=dev)
    tracer = W.PackedSDFTracer(num_steps=nsteps, step_size=step_size, min_dis=min_dis)
    pipe = W.Pipeline(nef, tracer)
    R = res * res
    total = args.warmup + args.steps
    from oracle import oracle as O
    cams = [O.look_at_rays(orbit_origin((i * world + rank) * 3), CAM_LOOKAT, res, res, CAM_FOV) for i in range(total)]
    cams = [(o * np.float32(0.75), d) for o, d in cams]                              # radius ~3.2: the sphere-like surface fills the frame
    host = [(torch.from_numpy(np.ascontiguousarray(o)).pin_memory(), torch.from_numpy(d).pin_memory()) for o, d in cams]
    devr = [(o.to(dev), d.to(dev)) for o, d in host]
    chans = ["rgb", "depth", "hit", "normal"]

    # parity on a 64^2 slice of the same model (rank 0): the numpy restatement pinned by tests/golden/sdf_octree.npz
    parity, cpu_base = None, None
    if rank == 0 and not args.no_cpu_baseline:
        t0 = time.perf_counter()
        ref = OG.sdf_trace(case, num_steps=nsteps, step_size=step_size, min_dis=min_dis, dist_max=6.0)
        dt = time.perf_counter() - t0
        with torch.no_grad():
            rb = pipe(rays=W.Rays(torch.from_numpy(case["origins"]).to(dev), torch.from_numpy(case["dirs"]).to(dev), 0.0, 6.0), channels=chans)
        hit = rb.hit.cpu().numpy(); both = hit & ref["hit"]
        parity = {"rays": int(hit.size), "hits_cpu": int(ref["hit"].sum()), "hit_flips": int((hit != ref["hit"]).sum()),
                  "depth_max_abs_err": float(np.abs(rb.depth.cpu().numpy()[both] - ref["depth"][both]).max()) if both.any() else 0.0,
                  "normal_min_dot": float((rb.normal.cpu().numpy()[both] * ref["normal"][both]).sum(-1).min()) if both.any() else 1.0,
                  "tolerance": {"hit_flips": "<= 0.2 %", "depth": 1e-4, "normal_dot": 0.99}}
        parity["ok"] = bool(parity["hit_flips"] <= max(1, hit.size // 500) and parity["depth_max_abs_err"] <= 1e-4 and parity["normal_min_dot"] >= 0.99)
        if not parity["ok"]:
            print(json.dumps({"parity_failure": parity}), file=sys.stderr, flush=True)
            raise SystemExit("bench.py --config 3: GPU sphere trace differs from the restatement beyond the stated tolerance")
        cpu_base = {"value": hit.size / dt, "unit": "rays/s", "cores": 1, "kind": "port",
                    "sample": f"{hit.size} rays (64^2 view of the same model), numpy restatement of packed_sdf_tracer.py:78-174 (single thread + OpenMP octree query), {dt:.2f} s"}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    # untimed setup: size the per-nugget buffers for the largest nugget count of this run's cameras (as reserve_samples does for the
    # radiance-field configurations); without it the caching allocator goes to cudaMalloc whenever a camera beats the previous maximum
    W.ops.reserve_nuggets(max(int(W.ops.raytrace(nef.grid.blas.tensors(), o_, d_, nef.grid.active_lods[-1])[0].shape[0]) for o_, d_ in devr))
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    with torch.no_grad():
        evals = []
        for i in range(args.warmup):       # same body as the timed loop (the previous frame's outputs stay alive while the next one renders): the
            rb = pipe(rays=W.Rays(*devr[i], 0.0, 6.0), channels=chans)       # caching allocator reaches its steady state before the timed region
            evals.append(tracer.prev_num_evals.clone())
        barrier()
        W.ops.PROFILE = []
        l0 = W._cabi.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        evals, hits = [], 0
        sev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
        dev_allocs0 = torch.cuda.memory_stats(dev).get("num_device_alloc", 0)
        e0.record(); sev[0].record()
        for k in range(args.steps):
            rb = pipe(rays=W.Rays(*devr[args.warmup + k], 0.0, 6.0), channels=chans)
            evals.append(tracer.prev_num_evals.clone())
            sev[k + 1].record()
            if args.trace_host:
                ms_ = torch.cuda.memory_stats(dev)
                print("step", k, "device allocs", ms_.get("num_device_alloc", 0), "reserved MB", ms_.get("reserved_bytes.all.current", 0) / 1e6, file=sys.stderr)
        e1.record()
        barrier()
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, host_arrays({c: getattr(rb, c) for c in chans}))
        step_ms3 = [sev[k].elapsed_time(sev[k + 1]) for k in range(args.steps)]
        dev_allocs3 = torch.cuda.memory_stats(dev).get("num_device_alloc", 0) - dev_allocs0
        launches = W._cabi.launch_count() - l0
        prof, W.ops.PROFILE = W.ops.PROFILE, None
        hits = int(rb.hit.sum())
        n_evals = float(sum(int(e) for e in evals))
        ms = e0.elapsed_time(e1)
        stage = {}
        for name, a, b in prof:
            stage.setdefault(name, []).append(a.elapsed_time(b))
        # end to end: rays from pinned host memory, the rgb + hit image read back
        e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        out_rgb = torch.empty((R, 3), dtype=torch.float32).pin_memory(); out_hit = torch.empty(R, dtype=torch.bool).pin_memory()
        for k in range(args.warmup):
            o, d = (t.to(dev, non_blocking=True) for t in host[k]); pipe(rays=W.Rays(o, d, 0.0, 6.0), channels=chans)
        barrier()
        e2.record()
        for k in range(args.steps):
            o, d = (t.to(dev, non_blocking=True) for t in host[args.warmup + k])
            rb = pipe(rays=W.Rays(o, d, 0.0, 6.0), channels=chans)
            out_rgb.copy_(rb.rgb, non_blocking=True); out_hit.copy_(rb.hit, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        e3.record()
        barrier()
        ms_e2e = e2.elapsed_time(e3)
    clocks = sampler.stop() if rank == 0 else None
    hbm, src = _peaks()

    def line(ms, ms_e2e, extra):
        ev = extra[0]
        t_trace = float(np.mean(stage.get("sdf_trace", [ms / args.steps])))
        per_eval = 6 * 8 * 16 * 2 + 6 * 8 * 4                                       # SURVEY 8(d): fp16-equivalent feature bytes + trinkets per LOD
        ach = (ev / (args.steps * world)) * per_eval / (t_trace * 1e-3) / 1e9
        return {"metric": "rays/sec sphere-trace 512^2 nglod OctreeGrid SDF (BASELINE config 3)", "value": R * args.steps * world / (ms * 1e-3), "unit": "rays/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32 decoder, f16-rounded octree features (octree_grid.py:147-149)", "data": "synthetic",
                "config": {"workload": f"app/nglod OctreeGrid level 7, F=16 x 6 LODs 'sum', NeuralSDF 19-128-1, PackedSDFTracer(32 steps, 0.8), {res}^2 rays, "
                                       "octahedron-shell octree (13 201 level-7 cells), orbit camera, render (no gradients: the tracer is inference-only)",
                           "rays_per_step_per_gpu": R, "l2": "a different camera every step; the feature levels (3 MB) are L2 resident by design",
                           "parallelism": f"dp{world} (one view per GPU, no collective)" if world > 1 else "single GPU"},
                "e2e": {"value": R * args.steps * world / (ms_e2e * 1e-3), "unit": "rays/s", "h2d_bytes_per_step": R * 24, "d2h_bytes_per_step": R * 13,
                        "ms_per_step": ms_e2e / args.steps},
                "gpu_launches": int(launches), "clocks": clocks,
                "roofline": _ncu_facts({"bound": "hbm", "kernel": "wb_sdf_trace_kernel", "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm, "traffic": None,
                             "kernel_ms": t_trace, "algorithmic_per_eval": f"{per_eval} B", "evals_per_launch": ev / (args.steps * world), "peak_source": src,
                             "note": "HBM-equivalent: the feature levels are L2 resident; the kernel is a latency chain of <= 33 dependent field evaluations per ray"},
                                       "wb_sdf_trace_kernel"),
                "stage_ms": {k: float(np.mean(v)) for k, v in stage.items()}, "hits_last_frame": hits, "field_evals_per_frame": ev / (args.steps * world),
                "step_ms": step_ms3, "cudaMalloc_calls_in_timed_region": int(dev_allocs3),
                "cpu_baseline": cpu_base, "parity": parity}
    _finish_line(args, torch, dist, world, rank, dev, line, ms, ms_e2e, [n_evals])


def run_config4(args):
    """One step = fwd + bwd + Adam on an 800^2 frame through Pipeline(NeuralRadianceField(TriplanarGrid fdim 4, 4 LODs 65^2..513^2,
    'sum'), PackedRFTracer('voxel', 512)) over an AABB (nerf_triplanar.yaml shapes with log_base_resolution 6): FUSED path."""
    import torch
    import torch.distributed as dist
    import wisp_b200 as W
    from oracle import oracle as O
    world, rank, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local); dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    res = 800 if args.res == 1024 else args.res
    nsteps = 512 if args.num_steps == 2048 else args.num_steps
    torch.manual_seed(0)
    blas = W.AxisAlignedBBoxAS(device=dev)
    grid = W.TriplanarGrid(blas, feature_dim=4, log_base_resolution=6, num_lods=4, multiscale_type='sum', feature_std=0.01)
    nef = W.NeuralRadianceField(grid, view_embedder='positional', view_multires=4, hidden_dim=64, num_layers=1, bias=True).to(dev)
    tracer = W.PackedRFTracer(raymarch_type='voxel', num_steps=nsteps, bg_color=(1.0, 1.0, 1.0)); tracer.precision = args.precision
    pipe = W.Pipeline(nef, tracer)
    params = [p for p in nef.parameters() if p.requires_grad]
    opt = torch.optim.Adam(params, lr=1e-3, eps=1e-15, fused=True)
    reducer = W.parallel.GradientReducer(params)
    R = res * res
    total = args.warmup + args.steps
    g = torch.Generator().manual_seed(2)
    host = []
    for i in range(total):
        o, d = O.look_at_rays(orbit_origin(i * world + rank), CAM_LOOKAT, res, res, CAM_FOV)
        host.append((torch.from_numpy(o).pin_memory(), torch.from_numpy(d).pin_memory(), torch.sigmoid(torch.randn(R, 3, generator=g)).pin_memory()))
    devb = [tuple(t.to(dev) for t in b) for b in host]

    # parity (rank 0): fused tensor-core path vs the unfused route (native triplane kernel pinned to the reference golden + torch decoders)
    parity = None
    if rank == 0 and not args.no_cpu_baseline:
        o, d, t = (x[:: max(1, R // 16384)][:16384].contiguous() for x in devb[0])
        outs = []
        for fused in (False, True):
            for p_ in params:
                p_.grad = None
            if not fused:
                nef.fused_spec = lambda lod_idx=None: None
            tracer.seed = 3
            tracer.precision = args.precision if fused else 0
            rb = pipe(rays=W.Rays(o, d, NEAR, FAR), channels=["rgb"])
            torch.nn.functional.smooth_l1_loss(rb.rgb, t).backward()
            outs.append((rb.rgb.detach().clone(), {n: p_.grad.clone() for n, p_ in nef.named_parameters() if p_.grad is not None}))
            if not fused:
                del nef.fused_spec
        tracer.precision = args.precision
        tol = dict(PARITY_TOL[int(args.precision)])
        if args.precision == 1:
            tol["grad"] = 8e-2       # 'sum' grid: every LOD receives the same dL/dfeat; coarse texels add ~10^5 signed fp16-carried terms
        gerr = max(float((outs[1][1][n] - gr).abs().max() / gr.abs().max().clamp_min(1e-30)) for n, gr in outs[0][1].items())
        parity = {"rays": int(o.shape[0]), "rgb_max_abs_err": float((outs[1][0] - outs[0][0]).abs().max()), "grad_max_rel_err": gerr, "tolerance": tol,
                  "checked_against": "unfused route: wb_triplane kernel (pinned to tests/golden/triplanar.npz) + torch nn.Linear decoders, fp32"}
        parity["ok"] = bool(parity["rgb_max_abs_err"] <= tol["rgb"] and gerr <= tol["grad"])
        for p_ in params:
            p_.grad = None
        if not parity["ok"]:
            print(json.dumps({"parity_failure": parity}), file=sys.stderr, flush=True)
            raise SystemExit("bench.py --config 4: fused path differs from the unfused route beyond the stated tolerance")

    last_rgb = [None]                      # --dump-outputs: the image of the latest step

    def step(i, o, d, t):
        opt.zero_grad(set_to_none=True)
        tracer.seed = 1000 + i * world + rank
        rb = pipe(rays=W.Rays(o, d, dist_min=NEAR, dist_max=FAR), channels=["rgb"])
        if args.dump_outputs:
            last_rgb[0] = rb.rgb.detach()
        loss = torch.nn.functional.smooth_l1_loss(rb.rgb, t, reduction='none').mean()
        loss.backward()
        reducer.reduce()
        opt.step()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    W.ops.reserve_samples(R * nsteps)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for i in range(args.warmup):
        step(i, *devb[i])
    barrier()
    W.ops.PROFILE = []
    l0 = W._cabi.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    S_total = 0
    e0.record()
    for k in range(args.steps):
        loss = step(args.warmup + k, *devb[args.warmup + k]); S_total += tracer.get_prev_num_samples()
    e1.record()
    barrier()
    if args.dump_outputs and rank == 0:   # before the e2e leg below takes further optimiser steps
        dump_outputs(args.dump_outputs, host_arrays({"loss": loss, "rgb": last_rgb[0], **dict(nef.named_parameters())}))
    launches = W._cabi.launch_count() - l0
    prof, W.ops.PROFILE = W.ops.PROFILE, None
    ms = e0.elapsed_time(e1)
    stage = {}
    for name, a, b in prof:
        stage.setdefault(name, []).append(a.elapsed_time(b))
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pre = W.parallel.HostPrefetcher(host[:args.warmup], dev)
    for k, b in enumerate(pre):
        step(k, *b)
    barrier()
    e2.record()
    last = None
    pre = W.parallel.HostPrefetcher(host[args.warmup:], dev)
    for k, b in enumerate(pre):
        last = float(step(args.warmup + k, *b).item())
    e3.record()
    barrier()
    ms_e2e = e2.elapsed_time(e3)
    clocks = sampler.stop() if rank == 0 else None
    hbm, src = _peaks()

    def line(ms, ms_e2e, extra):
        S_step = extra[0] / (args.steps * world)
        mean = {k: float(np.mean(v)) for k, v in stage.items()}
        per = 4 * 3 * 4 * 4 * 4                                                   # SURVEY 8(d): L * 3 planes * 4 texels * fdim * 4 B = 768 B/sample
        roofs = []
        for st_name, kern, mult in (("shade_fwd", "wb_shade_fwd_tc_kernel<GX>" if args.precision == 1 else "wb_shade_fwd_kernel", 1),
                                    ("table_scatter", "wb_featx_scatter_kernel", 2), ("decoder_bwd", "wb_mlp_bwd3_tc_kernel", 0)):
            if st_name in mean and mult:
                a = S_step * per * mult / (mean[st_name] * 1e-3) / 1e9
                roofs.append({"bound": "hbm", "kernel": kern, "achieved": a, "peak": hbm, "unit": "GB/s", "frac": a / hbm, "traffic": None,
                              "kernel_ms": mean[st_name], "algorithmic_per_sample": f"{per * mult} B", "samples_per_launch": S_step})
        roof = dict(max(roofs, key=lambda r: r["kernel_ms"])) if roofs else None
        if roof:
            roof["peak_source"] = src
            roof["note"] = "HBM-equivalent: the planes (12.6 MB) are L2 resident"
            _ncu_facts(roof, "wb_shade_fwd_tc_kernel_cfg4" if roof["kernel"].startswith("wb_shade_fwd_tc") else "wb_featx_scatter_kernel_cfg4")
        return {"metric": "rays/sec (fwd+bwd) 800^2 TriplanarGrid NeRF (BASELINE config 4)", "value": R * args.steps * world / (ms * 1e-3), "unit": "rays/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32" if args.precision == 0 else "f16(tensor)+f32 accumulate", "data": "synthetic",
                "config": {"workload": f"TriplanarGrid fdim 4, 4 LODs 65^2..513^2 'sum', 2-layer-64 MLP, AABB, 'voxel' {nsteps} steps, {res}^2 rays, fwd+bwd+Adam, fused path",
                           "rays_per_step_per_gpu": R, "l2": "per-step sample records + saved features (> 10 GB) exceed the 126 MB L2; a different camera every step",
                           "parallelism": f"dp{world} (one view per GPU per step, NCCL all-reduce of gradients)" if world > 1 else "single GPU"},
                "e2e": {"value": R * args.steps * world / (ms_e2e * 1e-3), "unit": "rays/s", "h2d_bytes_per_step": R * 36, "d2h_bytes_per_step": 4,
                        "ms_per_step": ms_e2e / args.steps, "last_loss": last},
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "rooflines": roofs, "stage_ms": mean,
                "samples_per_step_per_gpu": S_step, "samples_per_sec": extra[0] / (ms * 1e-3), "parity": parity,
                "cpu_baseline": None if args.no_cpu_baseline else {"value": None, "unit": "rays/s", "cores": 0, "kind": "port",
                                                                   "sample": "no CPU restatement of the triplanar field in oracle/ (torch F.grid_sample is the pin); see --config 2 for the CPU arm"}}
    _finish_line(args, torch, dist, world, rank, dev, line, ms, ms_e2e, [float(S_total)])



if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    elif a.config == 3:
        run_config3(a)
    elif a.config == 4:
        run_config4(a)
    else:
        run_ours(a)
