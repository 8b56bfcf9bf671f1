#!/usr/bin/env python
"""bench.py -- the metric of BASELINE.json on B200.

Workloads (`config.workload` names the BASELINE.json config each one is):
  default / --workload shapegen   configs[1] (and [2], [4] through the flags below): one "step" = one synthetic
      512x512 masked crop -> DINOv2 conditioner -> 50 CFG DiT steps -> ShapeVAE -> (R+1)^3 SDF decode -> marching
      cubes -> mesh.  --octree 512 is configs[4]'s grid; --objects N fixes the TOTAL number of objects and splits them
      over the ranks (strong scaling: configs[2] = --objects 8 on 8 GPUs, configs[4] = --objects 32 --octree 512).
  --workload vggt                 configs[3]: VGGT depth + camera forward (2 frames loaded at 1024^2, run at 518^2 as
      the reference stage does) + point-cloud back-projection; roofline = the back-projection kernel's HBM GB/s.

  python bench.py --gpus N --steps K --warmup W            # our arm (one rank per GPU under torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port) on the host cores

`value`  : objects/s with the preprocessed crop already resident in HBM and the mesh left on the device.
`e2e`    : objects/s through the public call `pipe(image=<PIL RGBA>, ..., output_type="mesh")` with host buffers: the
           image processor, the pinned host -> device copy of the crop and the device -> host landing of the mesh
           (pinned ring, r3g.dist.MeshStreamGatherer) are inside the timed region, every step.
On one GPU the two arms are INTERLEAVED object by object inside one barrier-bracketed region (device-resident object,
then end-to-end object, K times) and each arm's time is the sum of its own CUDA-event segments, so both see the same
clocks.  On N > 1 GPUs the arms run one after the other: the device-resident arm packs its meshes into a staging buffer and
moves them to rank 0 in one NCCL message per peer at the end (inside its timed region); the end-to-end arm does the same
and then lands every mesh in rank 0's pinned host ring (on one GPU each mesh streams there as it finishes, under the next
object's compute).
Objects are independent (src/2d_to_3d_models/run.py:188-193 shards them over GPUs): no data-path collective.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "3d-re-gen_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "objects->mesh/sec (256^3 SDF, 50 DiT steps)"
METRIC_VGGT = "VGGT depth+camera forward + point-cloud back-projection (frames/s; back-projection HBM GB/s vs peak)"


def workload_name(args):
    if args.workload == "vggt":
        return "VGGT depth+camera forward at 1024x1024 (run at 518x518 like the stage) + point-cloud back-projection"
    n = f"{args.objects} synthetic 512x512 masked crops" if args.objects else "single 512x512 masked crop"
    if getattr(args, "crops", "synthetic") == "2400":
        n = f"input_images/2400.jpg: {args.objects or 8} fixed-box object crops"
    return f"{n} -> Hunyuan3D-2 shape gen, {args.dit_steps} DiT steps, {args.octree}^3 SDF + marching cubes"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="r3g", choices=["r3g", "reference"])
    ap.add_argument("--workload", default="shapegen", choices=["shapegen", "vggt"])
    ap.add_argument("--octree", type=int, default=256)
    ap.add_argument("--dit-steps", type=int, default=50)
    ap.add_argument("--objects", type=int, default=0,
                    help="strong scaling: TOTAL objects, split over the ranks (overrides --steps)")
    ap.add_argument("--frames", type=int, default=2, help="vggt workload: frames per scene")
    ap.add_argument("--crops", default="synthetic", choices=["synthetic", "2400"],
                    help="2400: the 8 fixed-box crops of the reference's input_images/2400.jpg (BASELINE configs[2])")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-mode", action="store_true",
                    help="warm-up + device-resident loop only (for ncu launch lists); prints no bench line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/<name>.npy (float32 / float64; 64 MB in all, "
                         "a seeded sample of rows where an output is larger than its share), to compare two builds")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl r3g: the reference arm times bounded samples and keeps no outputs")
    return args


DUMP_BYTES = 60 << 20      # the arrays' data: with the .npy headers the files stay under 64 MB (64e6 bytes)


def dump_outputs(path, arrays):
    """--dump-outputs: every array as <path>/<name>.npy, float32 kept and any other dtype as float64.  The arrays share
    DUMP_BYTES equally; one larger than its share is viewed as rows of its last dimension and replaced by a fixed,
    seeded sample of those rows in their original order, so two builds that compute the same outputs write the same
    files."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    share = DUMP_BYTES // max(1, len(arrays))
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
        a = a.astype(np.float32 if a.dtype == np.float32 else np.float64)
        if a.nbytes > share:
            rows = a.reshape(-1, a.shape[-1])
            keep = share // rows[0].nbytes
            a = rows[np.sort(np.random.default_rng(0).choice(len(rows), keep, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(tflops=d.get("bf16_tflops_sustained", d.get("bf16_tflops")), hbm=d.get("hbm_gbs"),
                    source="MEASURED_PEAKS.json (sustained cuBLAS bf16; copy bandwidth)")
    return dict(tflops=1400.0, hbm=6650.0, source="fallback of B200_PROFILING.md")


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region."""

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = max((int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()), default=None)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower() == "active"})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons,
                "samples": len(sm)}


def host_threads():
    """Threads for the CPU arm: the physical cores.  torchrun exports OMP_NUM_THREADS=1 for nproc > 1 (round 1's arm
    slowed 9x exactly at N = 2), and one thread per LOGICAL core measured 4x slower than per physical core here
    (128 vs 64 on the r2b box: 8.5e-5 vs 3.5e-4 objects/s)."""
    try:
        import psutil
        n = psutil.cpu_count(logical=False)
    except Exception:
        n = None
    return int(n or max(1, (os.cpu_count() or 2) // 2))


def synthetic_crop(seed, size=512):
    """512x512 RGBA: uniform-noise RGB inside an elliptical alpha mask (SURVEY.md section 8d, config 2)."""
    import numpy as np
    from PIL import Image
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:size, 0:size]
    mask = (((xx - size / 2) / (0.38 * size)) ** 2 + ((yy - size / 2) / (0.30 * size)) ** 2) <= 1.0
    rgba = np.zeros((size, size, 4), np.uint8)
    rgba[..., :3] = rng.integers(0, 256, (size, size, 3), dtype=np.uint8)
    rgba[..., 3] = mask * 255
    return Image.fromarray(rgba, "RGBA")


def crops_2400():
    """tests/golden/crops_2400/*.jpg (tools/make_2400_crops.py) as RGBA with an opaque rectangular alpha."""
    from PIL import Image
    d = os.path.join(ROOT, "tests", "golden", "crops_2400")
    files = sorted(f for f in os.listdir(d) if f.endswith(".jpg"))
    return [Image.open(os.path.join(d, f)).convert("RGBA") for f in files]


def shapegen_config(args, world, per_rank):
    """The `config` object; both arms print exactly these keys for the same flags."""
    return {"workload": workload_name(args), "octree_resolution": args.octree, "dit_steps": args.dit_steps,
            "guidance": 5.0, "objects_per_gpu": per_rank, "objects_total": per_rank * world,
            "l2": "working set (2.6 GB of weights + a 68-540 MB grid per object) exceeds L2",
            "parallelism": f"objects sharded over {world} GPU(s), meshes gathered to rank 0 over NCCL"}


def reference_arm(args):
    """The reference's own CPU implementation of the path (oracle port, fp32 torch + C marching cubes) on ALL host
    cores.  torchrun exports OMP_NUM_THREADS=1 for nproc > 1: the thread count is set explicitly here, otherwise the
    arm slows 9x exactly when N >= 2 (round 1's void SCALE ratios)."""
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    torch.set_num_threads(host_threads())
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import cpu_baseline
    vals, det = [], None
    # every step is one bounded sample; with many steps the repetitions inside a sample shrink so that the whole arm
    # stays within a few minutes (>= 3 block timings enter the mean either way)
    reps = 3 if args.steps < 8 else 1
    for i in range(args.warmup + args.steps):
        if args.workload == "vggt":
            v, det = cpu_baseline.time_vggt_sample(args.frames, reps=reps)
        else:
            v, det = cpu_baseline.time_object_sample(args.octree, args.dit_steps, mc_grid=97, dit_reps=reps,
                                                     chunk_reps=max(1, reps - 1))
        if i >= args.warmup:
            vals.append(v)
    value = sum(vals) / len(vals)
    vggt = args.workload == "vggt"
    per_rank = (args.objects // world) if args.objects else args.steps
    cfg = ({"workload": workload_name(args), "frames": args.frames} if vggt else shapegen_config(args, world, per_rank))
    cfg["note"] = "each step times a bounded sample of the workload on the host cores and extrapolates linearly"
    line = {"metric": METRIC_VGGT if vggt else METRIC, "value": value, "unit": "frames/s" if vggt else "objects/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 / value,
            "higher_is_better": True, "scaling": "strong" if args.objects else "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "impl": "reference", "config": cfg,
            "cpu_baseline": {"value": value, "unit": "frames/s" if vggt else "objects/s",
                             "cores": torch.get_num_threads(), "kind": "port", "sample": det["sample"]},
            "e2e": {"value": value, "unit": "frames/s" if vggt else "objects/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# DRAM traffic of the DiT forward's GEMM launches: `ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum` over one
# forward (tools/prof_dit_gemm.py), averaged per launch like `achieved`; the committed capture is named beside it.
GEMM_TRAFFIC_NCU = {"source": "profiles/r2d_ncu_dit_gemm_traffic.csv.gz (131 launches of one forward, cold L2 per launch "
                              "under ncu: an upper bound of the in-graph traffic)",
                    "dram_bytes_per_launch": 85.34e6}


def instrumented_linear_roofline(pipe, cond, peak_tflops):
    """Dominant kernel = the tcgen05 GEMM (every nn.Linear of the DiT: ~46 % of the step in the ncu launch list).
    Its launches are isolated from the other kernels of the forward -- same weights, same order, same shapes and
    epilogues -- by recording one eager forward's r3g_linear calls and re-issuing exactly those into a CUDA graph,
    replayed between CUDA events on the launching stream.  achieved = sum of 2*M*N*K over the launches / elapsed."""
    import torch
    from r3g import ops
    calls = []          # (function, args, kwargs) of every GEMM launch of one forward, in order
    orig, orig_pair = ops.linear, ops.linear_pair

    def record(x, w, bias=None, **kw):
        calls.append((orig, (x, w, bias), kw))
        return orig(x, w, bias, **kw)

    def record_pair(first, second):
        calls.append((orig_pair, (first, second), {}))
        return orig_pair(first, second)

    x = torch.randn(2, pipe.vae.latent_shape[0], pipe.vae.latent_shape[1], device="cuda").half()
    t = torch.full((2,), 0.5, device="cuda", dtype=torch.float16)
    ops.linear, ops.linear_pair = record, record_pair
    try:
        pipe.model(x, t, cond)
    finally:
        ops.linear, ops.linear_pair = orig, orig_pair
    torch.cuda.synchronize()

    def rows(t_):
        return t_.numel() // t_.shape[-1]

    def problems(fn, a):
        return [(a[0], a[1])] if fn is orig else [(d["x"], d["w"]) for d in a]
    probs = [pw for fn, a, _ in calls for pw in problems(fn, a)]
    flops = sum(2.0 * rows(cx) * cw.shape[0] * cw.shape[1] for cx, cw in probs)
    alg_bytes = sum(2.0 * (rows(cx) * cw.shape[1] + cw.shape[0] * cw.shape[1] + rows(cx) * cw.shape[0]) for cx, cw in probs)
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for fn, a, kw in calls:
            fn(*a, **kw)
    torch.cuda.current_stream().wait_stream(side)
    with torch.cuda.graph(g):
        for fn, a, kw in calls:
            fn(*a, **kw)
    for _ in range(3):
        g.replay()
    reps = 5
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        g.replay()
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / reps
    achieved = flops / ms / 1e9
    return {"bound": "tensor", "kernel": "linear_kernel / linear_kernel_2cta (tcgen05 GEMM, gemm.cu): the DiT forward's launches",
            "launches_timed": len(calls), "gemm_problems": len(probs), "achieved": achieved, "peak": peak_tflops, "unit": "TFLOP/s",
            "frac": achieved / peak_tflops, "traffic": GEMM_TRAFFIC_NCU["dram_bytes_per_launch"],
            "traffic_source": GEMM_TRAFFIC_NCU["source"], "avg_launch_ms": ms / len(calls),
            "flops_per_launch_avg": flops / len(calls), "algorithmic_bytes_per_launch_avg": alg_bytes / len(calls),
            "note": "weights stream from HBM (2.2 GB per forward > L2); activations mostly L2-resident, so DRAM traffic "
                    "per launch sits below the algorithmic bytes"}


def setup_dist():
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    if world > 1:
        dist.barrier()
    return world, rank, local


def main_shapegen(args):
    import torch
    import torch.distributed as dist

    world, rank, local = setup_dist()
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run")
    from r3g import _abi
    from r3g.dist import MeshBatchGatherer, MeshStreamGatherer
    from r3g.pipelines import Hunyuan3DDiTFlowMatchingPipeline

    pk = peaks()
    pipe = Hunyuan3DDiTFlowMatchingPipeline.from_random(seed=0, device=f"cuda:{local}")
    pipe.vae.surface_extractor.keep_on_device = True
    ctx = _abi.get_context(local)
    R = args.octree
    if args.objects:
        if args.objects % world:
            raise SystemExit(f"--objects {args.objects} must be a multiple of the {world} ranks")
        K = args.objects // world
    else:
        K = args.steps
    W = args.warmup

    # synthetic inputs: distinct crops per rank and arm; the device-resident arm gets them preprocessed and uploaded
    n_in = W + 2 * K
    if args.crops == "2400":        # object j of the scene goes to rank j % world (src/2d_to_3d_models/run.py:188-193)
        real = crops_2400()
        crops = [real[(rank + world * i) % len(real)] for i in range(n_in)]
    else:
        crops = [synthetic_crop(1234567 + rank * 1000 + i) for i in range(n_in)]
    dev_in = [pipe.image_processor(c)["image"].cuda() for c in crops]
    kw = dict(num_inference_steps=args.dit_steps, octree_resolution=R, num_chunks=16000, output_type="mesh")

    def object_resident(i):
        cond = pipe.encode_cond(dev_in[i], {}, True)
        return pipe(cond=cond, generator=torch.manual_seed(1234567 + i), **kw)[0]

    def object_e2e(i):
        """The call a user of the reference makes (src/2d_to_3d_models/run.py:77-84)."""
        return pipe(image=crops[i], generator=torch.manual_seed(1234567 + i), **kw)[0]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # warm-up (captures the DiT CUDA graph; sizes the gather capacity; lets the caching allocator see its blocks)
    warm = [object_resident(i) if i % 2 == 0 else object_e2e(i) for i in range(W)]
    ok = [m for m in warm if m is not None]
    cap_v = int(1.3 * max((m.mesh_v.shape[0] for m in ok), default=1)) + 1024
    cap_f = int(1.3 * max((m.mesh_f.shape[0] for m in ok), default=1)) + 1024
    del warm, ok
    d2h_bytes = [0]

    def count(step, r, v, f):          # consumer thread of the e2e gatherer on rank 0: bytes that landed on the host
        d2h_bytes[0] += v.numel() * 4 + f.numel() * 4
    # device-resident arm at N > 1: meshes are packed into a per-rank staging buffer and moved to rank 0 in ONE message
    # per peer at the end of the arm (no NCCL kernel is resident while objects compute); e2e arm: per-object streaming
    # gather on a side stream into rank 0's pinned ring
    # (one GPU: each mesh streams to the pinned host ring as it finishes, under the next object's compute).  A per-object
    # NCCL exchange during compute cost ~0.15 s per object at N = 8 (profiles/README.md r2d), so at N > 1 BOTH arms
    # keep NVLink quiet while objects compute and pay the gather -- and, for e2e, the pinned D2H of all meshes on rank 0 --
    # once, inside their timed regions.
    g_dev = MeshBatchGatherer(cap_v, cap_f, K, f"cuda:{local}") if world > 1 else None
    g_e2e = (MeshBatchGatherer(cap_v, cap_f, K, f"cuda:{local}", to_host=True) if world > 1
             else MeshStreamGatherer(cap_v, cap_f, device=f"cuda:{local}", to_host=True, sink=count))
    interleave = world == 1            # one GPU: the two arms alternate object by object and see the same clocks

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    launches0 = ctx.launches + pipe.replayed_launches
    h2d = 0
    meshes = []
    kept = {}                          # --dump-outputs: the meshes of the last timed step
    seg_dev, seg_e2e = [], []

    def mark():
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def do_resident(k):
        a = mark()
        m = object_resident(W + 2 * k)
        if g_dev is not None:
            g_dev.submit(*((m.mesh_v, m.mesh_f) if m is not None else (None, None)))
        seg_dev.append((a, mark()))
        if k == 0:      # only the first mesh is kept (for the line's statistics): holding all K would make every later
            meshes.append(m)    # object cudaMalloc fresh ~200 MB blocks (100 ms each) inside the timed region
        if args.dump_outputs and k == K - 1:
            kept["resident"] = m

    host = {"pipe_call_ms": 0.0, "gather_submit_ms": 0.0}      # host wall time of the two halves of an e2e step

    def do_e2e(k):
        nonlocal h2d
        a = mark()
        t0 = time.perf_counter()
        m2 = object_e2e(W + 2 * k + 1)
        t1 = time.perf_counter()
        h2d += dev_in[0].numel() * 4
        g_e2e.submit(*((m2.mesh_v, m2.mesh_f) if m2 is not None else (None, None)))
        host["pipe_call_ms"] += 1e3 * (t1 - t0) / K
        host["gather_submit_ms"] += 1e3 * (time.perf_counter() - t1) / K
        seg_e2e.append((a, mark()))
        if args.dump_outputs and k == K - 1:
            kept["e2e"] = m2

    barrier()
    if args.profile_mode:
        torch.cuda.nvtx.range_push("timed")      # ncu --nvtx --nvtx-include "timed/" profiles the timed object(s) only
    if interleave:
        for k in range(K):
            do_resident(k)
            if not args.profile_mode:
                do_e2e(k)
    else:
        for k in range(K):
            do_resident(k)
    if args.profile_mode:
        torch.cuda.synchronize()
        torch.cuda.nvtx.range_pop()
    a = mark()
    if g_dev is not None:
        g_dev.finish()                  # one NCCL message per peer: every rank's K meshes are on rank 0's device
    seg_dev.append((a, mark()))
    if not interleave and not args.profile_mode:
        barrier()
        for k in range(K):
            do_e2e(k)
    a = mark()
    if world > 1:
        g_e2e.finish(to_host=True, sink=count)   # every rank's meshes gathered to rank 0 and landed in its pinned ring
    else:
        g_e2e.finish()                  # the last object's mesh has landed on rank 0's host
    seg_e2e.append((a, mark()))
    barrier()
    clk = clocks.stop() if rank == 0 else None
    ms_dev = sum(x.elapsed_time(y) for x, y in seg_dev)
    ms_e2e = sum(x.elapsed_time(y) for x, y in seg_e2e)
    launches = (ctx.launches + pipe.replayed_launches - launches0)
    t = torch.tensor([ms_dev, ms_e2e], device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_dev, ms_e2e = t.tolist()
    stage = dict(pipe.timings)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {f"{arm}_mesh_{part}": getattr(m, attr)
                                         for arm, m in kept.items() if m is not None
                                         for part, attr in (("vertices", "mesh_v"), ("faces", "mesh_f"))})
    if args.profile_mode:
        if rank == 0:
            print(json.dumps({"profile_mode": True, "ms_per_step": ms_dev / K, "stages_ms_last_object": stage}))
        return
    value = world * K / (ms_dev / 1000.0)
    e2e_value = world * K / (ms_e2e / 1000.0)
    if rank == 0:
        cond = pipe.encode_cond(dev_in[0], {}, True)
        roof = instrumented_linear_roofline(pipe, cond, pk["tflops"])
        roof["peak_source"] = pk["source"]
        # whole-step view: algorithmic FLOPs of one object (SURVEY.md section 8d) over the measured step time
        Li, Lt = pipe.vae.latent_shape[0], cond["main"].shape[1]
        fl_obj = (2 * args.dit_steps * pipe.model.flops_per_sample(Li, Lt) + pipe.vae.flops_forward()
                  + (R + 1) ** 3 * pipe.vae.geo_decoder.flops_per_query(Li))
        m0 = meshes[0]
        line = {
            "metric": METRIC, "value": value, "unit": "objects/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": "strong" if args.objects else "weak",
            "vs_baseline": None, "dtype": "f16",
            "data": ("synthetic (seeded random weights of the Hunyuan3D-2 architecture; "
                     + ("fixed-box crops of input_images/2400.jpg)" if args.crops == "2400" else "noise crops)")),
            "config": shapegen_config(args, world, K),
            "e2e": {"value": e2e_value, "unit": "objects/s", "h2d_bytes_per_step": h2d // K,
                    "d2h_bytes_per_step": d2h_bytes[0] // (K * world) if world > 1 else d2h_bytes[0] // K,
                    "d2h_bytes_total_on_rank0": d2h_bytes[0], "ms_per_step": ms_e2e / K, "host_ms_per_step": host,
                    "call": "pipe(image=<PIL RGBA>, ..., output_type='mesh') + mesh landed in pinned host memory on rank 0"},
            "gpu_launches": int(launches),
            "clocks": clk,
            "roofline": roof,
            "stages_ms_last_object": stage,
            "object": {"algorithmic_tflop": fl_obj / 1e12,
                       "achieved_tflops_whole_step": fl_obj / 1e12 / (ms_dev / K / 1e3),
                       "frac_of_peak_whole_step": fl_obj / 1e12 / (ms_dev / K / 1e3) / pk["tflops"],
                       "mesh_vertices": int(m0.mesh_v.shape[0]) if m0 is not None else 0,
                       "mesh_faces": int(m0.mesh_f.shape[0]) if m0 is not None else 0},
        }
        if not args.no_cpu_baseline and world == 1:
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            import cpu_baseline
            torch.set_num_threads(host_threads())
            v, det = cpu_baseline.time_object_sample(R, args.dit_steps)
            line["cpu_baseline"] = {"value": v, "unit": "objects/s", "cores": torch.get_num_threads(), "kind": "port",
                                    "sample": det["sample"], "sampled_cpu_seconds": det["sampled_cpu_seconds"],
                                    "extrapolated_object_s": det["extrapolated_object_s"]}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main_vggt(args):
    """configs[3].  One step = one scene: S frames (host tensors [S,3,1024,1024], the reference's load resolution) ->
    bilinear resize to 518 -> aggregator (r3g kernels) -> camera head -> DPT depth head -> r3g_unproject (float64)."""
    import importlib.util
    import numpy as np
    import torch
    import torch.distributed as dist

    world, rank, local = setup_dist()
    from r3g import _abi, ops
    from r3g.vggt_heads import VGGT, random_state_dict
    spec = importlib.util.spec_from_file_location(
        "stage4", os.path.join(ROOT, "stages", "camera_and_pointcloud", "minimal_demo_vggt.py"))
    stage4 = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(stage4)
    pk = peaks()
    ctx = _abi.get_context(local)
    model = VGGT(device=f"cuda:{local}").load_state_dict(random_state_dict(0))
    S, K, W = args.frames, args.steps, args.warmup
    g = torch.Generator().manual_seed(1234567 + rank)
    host_in = [torch.rand(S, 3, 1024, 1024, generator=g).pin_memory() for _ in range(K + W)]
    dev_in = [h.cuda() for h in host_in]
    host_pts = torch.empty(S, 518, 518, 3, dtype=torch.float64).pin_memory()
    host_dc = torch.empty(2, S, 518, 518, dtype=torch.float32).pin_memory()

    def scene(images):
        E, Kmat, depth, conf = stage4.run_VGGT(model, images, 518)
        pts = ops.unproject(depth[..., 0].contiguous(), E, Kmat, torch.float64)
        return pts, depth, conf

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for i in range(W):
        scene(dev_in[i])
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * K + 1)]
    launches0 = ctx.launches
    h2d = d2h = 0
    barrier()
    ev[0].record()
    kept = {}                          # --dump-outputs: what the last timed step's device-resident scene returned
    for k in range(K):
        res = scene(dev_in[W + k])
        if args.dump_outputs and k == K - 1:
            kept = dict(zip(("resident_points", "resident_depth", "resident_conf"), res))
        del res
        ev[2 * k + 1].record()
        img = host_in[W + k].cuda(non_blocking=True)
        h2d += host_in[W + k].numel() * 4
        pts, depth, conf = scene(img)
        host_pts.copy_(pts, non_blocking=True)
        host_dc[0].copy_(depth[..., 0], non_blocking=True)
        host_dc[1].copy_(conf, non_blocking=True)
        d2h += host_pts.numel() * 8 + host_dc.numel() * 4
        ev[2 * k + 2].record()
    barrier()
    clk = clocks.stop() if rank == 0 else None
    launches = ctx.launches - launches0
    ms_dev = sum(ev[2 * k].elapsed_time(ev[2 * k + 1]) for k in range(K))
    ms_e2e = sum(ev[2 * k + 1].elapsed_time(ev[2 * k + 2]) for k in range(K))
    t = torch.tensor([ms_dev, ms_e2e], device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_dev, ms_e2e = t.tolist()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(kept, e2e_points=host_pts, e2e_depth=host_dc[0], e2e_conf=host_dc[1]))
    if rank == 0:
        # roofline: the back-projection kernel on a shape long enough to read a bandwidth (SURVEY.md section 8d row 4:
        # the real 2 x 518^2 call is 8.6 MB = launch-latency bound)
        rng = np.random.default_rng(0)
        Sx, H, Wd = 64, 1022, 1022
        dm = torch.rand(Sx, H, Wd, device="cuda") + 0.5
        q, _ = np.linalg.qr(rng.normal(size=(3, 3)))
        E = np.tile(np.concatenate([q, rng.normal(size=(3, 1))], 1).astype(np.float32), (Sx, 1, 1))
        Km = np.tile(np.array([[800, 0, 511], [0, 800, 511], [0, 0, 1]], np.float32), (Sx, 1, 1))
        out = torch.empty(Sx, H, Wd, 3, device="cuda", dtype=torch.float64)     # 1.6 GB, written in full by every launch
        for _ in range(3):
            ops.unproject(dm, E, Km, torch.float64, out=out)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 10
        a.record()
        for _ in range(reps):
            ops.unproject(dm, E, Km, torch.float64, out=out)
        b.record()
        torch.cuda.synchronize()
        ms_u = a.elapsed_time(b) / reps
        alg = Sx * H * Wd * (4 + 24)
        # aggregator alone, for the tensor-pipe view
        imgs518 = torch.nn.functional.interpolate(dev_in[0], size=(518, 518), mode="bilinear", align_corners=False)[None]
        for _ in range(2):
            model.aggregator(imgs518)
        a.record()
        for _ in range(5):
            model.aggregator(imgs518)
        b.record()
        torch.cuda.synchronize()
        ms_agg = a.elapsed_time(b) / 5
        P, C, depth_n = 1374, 1024, 24
        fl = S * P * 24 * C * C * 72 + 4 * C * (24 * S * P * P + depth_n * S * P * P + depth_n * (S * P) ** 2)
        line = {"metric": METRIC_VGGT, "value": world * K * S / (ms_dev / 1000.0), "unit": "frames/s", "n_gpus": world,
                "steps": K, "warmup": W, "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f16 operands / f32 residual stream (aggregator), f32 heads, f64 back-projection",
                "data": "synthetic (seeded random weights of the VGGT-1B camera+depth architecture; uniform-noise frames)",
                "config": {"workload": workload_name(args), "frames": S, "resolution": 518, "load_resolution": 1024,
                           "l2": "1.2 B parameters (2.4 GB fp16 + fp32 heads) exceed L2",
                           "parallelism": f"{world} independent replica(s): one forward per scene does not shard (DESIGN.md section 5)"},
                "e2e": {"value": world * K * S / (ms_e2e / 1000.0), "unit": "frames/s", "h2d_bytes_per_step": h2d // K,
                        "d2h_bytes_per_step": d2h // K, "ms_per_step": ms_e2e / K},
                "gpu_launches": int(launches), "clocks": clk,
                "roofline": {"bound": "hbm", "kernel": "unproject_kernel<f64> (rowops.cu) on [64,1022,1022]",
                             "achieved": alg / ms_u / 1e6, "peak": pk["hbm"], "unit": "GB/s",
                             "frac": alg / ms_u / 1e6 / pk["hbm"], "traffic": None, "avg_launch_ms": ms_u,
                             "algorithmic_bytes_per_launch": alg, "peak_source": pk["source"],
                             "note": "4 B read + 24 B written per pixel; the real 2x518x518 call moves 15 MB (launch bound)"},
                "aggregator": {"ms": ms_agg, "algorithmic_tflop": fl / 1e12, "tflops": fl / ms_agg / 1e9,
                               "frac_of_tensor_peak": fl / ms_agg / 1e9 / pk["tflops"]}}
        del out
        if not args.no_cpu_baseline and world == 1:
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            import cpu_baseline
            torch.set_num_threads(host_threads())
            v, det = cpu_baseline.time_vggt_sample(S, reps=3)
            line["cpu_baseline"] = {"value": v, "unit": "frames/s", "cores": torch.get_num_threads(), "kind": "port",
                                    "sample": det["sample"], "sampled_cpu_seconds": det["sampled_cpu_seconds"]}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        return reference_arm(args)
    if args.workload == "vggt":
        return main_vggt(args)
    return main_shapegen(args)


if __name__ == "__main__":
    main()
