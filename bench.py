#!/usr/bin/env python
"""bench.py — headline benchmark of the B200 wavefront path tracer.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run)
    python bench.py --impl reference --gpus N --steps K --warmup W

Workload (BASELINE.json configs[2], the one `metric` is quoted on): Sponza 1920x1080, depth 12, NEE+MIS,
HDR environment, frames x 1 spp.  The Khronos Sponza asset is not available offline, so the seeded
stand-in SURVEY.md §8d specifies is used: SynthSponza (seed 1234, 262 144 instanced triangles,
25 materials, 2048^2 sRGB/MR/normal value-noise textures, 10 % alpha-MASK foliage) + std_env.hdr.
One step = one frame = one pass of the hot path (ray-gen -> [traverse -> shade -> shadow/RR] x depth
-> accumulate) over every pixel of the framebuffer.

Numbers on the JSON line
  value          Mray/s, whole job, device-timed (CUDA events on the renderer's stream, max over ranks),
                 scene/BVH/textures/environment already resident in HBM.
  e2e            same metric through the public API with host buffers: every step passes the frame's
                 SceneFrameInfo + push constants from host memory and reads the RGBA32F accumulation
                 image back into pinned host memory.
  roofline       dominant kernel: algorithmic bytes (SURVEY.md §8d / DESIGN.md) / measured kernel time
                 vs the measured HBM peak in MEASURED_PEAKS.json.
  cpu_baseline   the CPU oracle (scalar port of the reference algorithm) on a bounded row band of the
                 same frame, all host threads.
N > 1: the framebuffer is tiled by rows (one strip per rank, scene replicated), one NCCL all-gather of
the strips per frame; total work is fixed, so scaling is "strong".
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "Mray/s @1080p SynthSponza (Sponza stand-in), depth 12, NEE+MIS, HDR env"  # config 3; CONFIG_SCENES has the others
NODE_BYTES, TRI_BYTES = 80, 48
DUMP_BYTES = 64_000_000  # --dump-outputs limit


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=3, choices=[2, 3, 4, 5],
                    help="BASELINE.json config (1-based like SURVEY.md section 8d): 3 = Sponza 1080p depth 12 (the headline metric, default), "
                         "2 = DamagedHelmet-class 1080p depth 8, 4 = DragonDispersion-class glass 1080p depth 32, 5 = Sponza 3840x2160 (8 ranks)")
    ap.add_argument("--width", type=int, default=0)
    ap.add_argument("--height", type=int, default=0)
    ap.add_argument("--depth", type=int, default=0)
    ap.add_argument("--omm", type=int, default=int(os.environ.get("B200PT_BENCH_OMM", "0")),
                    help="bake opacity micromaps of this subdivision level for the alpha-MASK triangles of the scene (0 = the asset as it is, without)")
    ap.add_argument("--no-omm-pass", action="store_true", help="skip the extra timed pass with baked opacity micromaps (configs 3 / 5, --omm 0)")
    ap.add_argument("--tex", type=int, default=2048)
    ap.add_argument("--detail", type=float, default=1.0)
    ap.add_argument("--cpu-rows", type=int, default=0, help="rows of the frame the CPU baseline renders (0 = sized for ~12 s)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-only", action="store_true", help="warm-up + K steps only (for runs under ncu); prints no bench line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the RGBA32F accumulation image they left (the image a caller reads back) to "
                         "DIR/accum.npy, every k-th row only where the whole image would exceed 64 MB (--impl ours)")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes what the CUDA path computed: use it with --impl ours")
    w, h, d = {2: (1920, 1080, 8), 3: (1920, 1080, 12), 4: (1920, 1080, 32), 5: (3840, 2160, 12)}[a.config]
    a.width, a.height, a.depth = a.width or w, a.height or h, a.depth or d
    return a


CONFIG_SCENES = {
    2: ("SynthHelmet(seed=1234): 46 080-triangle single mesh, one material with base colour / metallic-roughness / normal / emissive textures "
        "(stand-in for DamagedHelmet)", "Mray/s @1080p SynthHelmet (DamagedHelmet stand-in), depth 8, NEE+MIS, HDR env"),
    3: ("SynthSponza(seed=1234) stand-in for Sponza", "Mray/s @1080p SynthSponza (Sponza stand-in), depth 12, NEE+MIS, HDR env"),
    4: ("SynthGlass(seed=1234): 399 424-triangle displaced sphere, transmission 1, thickness 1, attenuationDistance 0.5, dispersion 20 "
        "(stand-in for DragonDispersion)", "Mray/s @1080p SynthGlass (DragonDispersion stand-in), depth 32, NEE+MIS, HDR env"),
    5: ("SynthSponza(seed=1234) stand-in for Sponza", "Mray/s @2160p SynthSponza (Sponza stand-in), depth 12, NEE+MIS, HDR env"),
}


def build_workload(args):
    """The synthetic scenes are deterministic in (seed, tex, detail); the generated arrays are cached as a pickle under
    the system temp dir so the N=1,2,4,8 and reference-arm invocations on one box generate them once."""
    import pickle
    from vk_gltf_renderer_b200 import hdr, synth
    env = hdr.load_hdr(os.path.join(ROOT, "tests", "assets", "std_env.hdr"))
    cfg = getattr(args, "config", 3)
    name = {2: "synthhelmet", 3: "synthsponza", 4: "synthglass", 5: "synthsponza"}[cfg]
    cache = os.path.join(tempfile.gettempdir(), "b200pt_%s_s1234_t%d_d%g.pkl" % (name, args.tex, args.detail))
    rank = int(os.environ.get("RANK", "0"))
    scn = None
    if os.path.exists(cache):
        try:
            with open(cache, "rb") as f:
                scn = synth.scene_from_state(pickle.load(f))
        except Exception:
            scn = None
    if scn is None:
        if cfg == 2:
            scn = synth.synth_helmet(seed=1234, tex_size=args.tex)
        elif cfg == 4:
            scn = synth.synth_glass(seed=1234, n=632, dispersion=20.0)
        else:
            scn = synth.synth_sponza(seed=1234, tex_size=args.tex, detail=args.detail)
        if rank == 0:
            try:
                tmp = cache + ".%d.tmp" % os.getpid()
                with open(tmp, "wb") as f:
                    pickle.dump(synth.scene_state(scn), f, protocol=4)
                os.replace(tmp, cache)
            except Exception:
                pass
    scn.omm_stats = None
    if getattr(args, "omm", 0) > 0:
        # the offline bake an asset with EXT_mesh_opacity_micromap went through (vk_gltf_renderer_b200/omm.py); untimed, like scene loading
        from vk_gltf_renderer_b200 import omm
        scn.omm_stats = omm.bake_opacity_micromaps(scn, level=args.omm)
    return scn, env


def workload_config(args, scn, n_gpus):
    return {"workload": "%s, %dx%d, depth %d, 1 spp/frame, std_env.hdr, NEE+MIS"
                        % (CONFIG_SCENES[getattr(args, "config", 3)][0], args.width, args.height, args.depth),
            "baseline_config": getattr(args, "config", 3),
            "triangles": scn.num_triangles(), "materials": len(scn.materials), "textures": len(scn.textures),
            "texture_size": args.tex, "opacity_micromaps": getattr(scn, "omm_stats", None), "partition": "1 GPU" if n_gpus == 1 else "interleaved row bands x%d, scene replicated; %d consecutive frames run as one wavefront per rank (b200pt_set_frame_batch) "
                         "and ONE NCCL all-gather of the RGBA32F tiles per batch (accumulation is linear: SURVEY.md section 8e)" % (n_gpus, n_gpus),
            "l2_policy": "no explicit flush: every frame streams its lane's path state (248 B x %d paths per rank = %.0f MB) plus the %.0f MB image, "
                         "and consecutive frames use different lanes; the working set exceeds the 126 MB L2 for N <= 4 "
                         "(at N = 8 a rank's 64 MB tile state would fit, its 8 lanes together do not)"
                         % (args.width * args.height // n_gpus, 248e-6 * args.width * args.height / n_gpus, 16e-6 * args.width * args.height)}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            self.path = tempfile.mktemp(suffix=".csv")
            q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.proc:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(smax)), reasons=sorted(reasons), samples=len(sm))
        try:
            os.unlink(self.path)
        except OSError:
            pass
        return out


def usable_cores():
    """Host cores this process may actually use: the scheduler affinity capped by the cgroup CPU quota (the GPU boxes show
    128 CPUs but a 16-core quota; 128 threads then run slower than 32)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(-(-int(quota) // int(period)))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, -(-q // per)))
        except Exception:
            pass
    return n


def cpu_baseline(args, scn, env, oracle=None, frame=0):
    """Oracle (port of the reference algorithm) on a row band in the middle of the frame, all host threads."""
    from oracle import oracle as O
    from vk_gltf_renderer_b200 import camera as cm
    if oracle is None:
        oracle = O.Oracle()
        oracle.set_scene(scn)
        oracle.set_environment(env)
    quota = usable_cores()
    threads = min(os.cpu_count() or 1, 2 * quota)  # measured on the box: 16-core quota -> 32 threads fastest (64 same, 128 slower)
    fi = cm.make_frame_info(scn.camera, args.width, args.height)
    pc = cm.make_push_constant(scn.camera, args.height, frame_count=frame, total_samples=0, max_depth=args.depth)
    rows = args.cpu_rows
    if rows <= 0:
        # size the band for ~12 s of CPU work from a 8-row probe
        probe = np.zeros((8, args.width, 4), np.float32)
        t0 = time.perf_counter()
        oracle.render_frame(fi, pc, probe, y0=args.height // 2, rows=8, threads=threads)
        per_row = (time.perf_counter() - t0) / 8
        rows = int(max(8, min(args.height, 12.0 / max(per_row, 1e-6))))
        args.cpu_rows = rows
    rows = min(rows, args.height)
    y0 = (args.height - rows) // 2
    accum = np.zeros((rows, args.width, 4), np.float32)
    oracle.reset_stats()
    t0 = time.perf_counter()
    oracle.render_frame(fi, pc, accum, y0=y0, rows=rows, threads=threads)
    dt = time.perf_counter() - t0
    st = oracle.stats()
    rays = st["closestRays"] + st["shadowRays"]
    return oracle, {"value": rays / dt / 1e6, "unit": "Mray/s", "cores": threads, "cpu_quota_cores": quota, "kind": "port",
                    "sample": "rows %d..%d of frame %d (%d paths, %d rays, %.1f s)" % (y0, y0 + rows - 1, frame, rows * args.width, rays, dt),
                    "spp_per_s_full_frame": (rows / args.height) / dt}, dt, rays


def run_reference(args, emit):
    """--impl reference: the reference's own algorithm on the host cores (oracle port: the Vulkan-RT
    reference cannot be built or run here — DESIGN.md §Oracle)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    scn, env = build_workload(args)
    oracle = None
    for w in range(args.warmup):
        oracle, _, _, _ = cpu_baseline(args, scn, env, oracle, frame=w)
    tot_t = tot_r = 0.0
    cb = None
    for k in range(args.steps):
        oracle, cb, dt, rays = cpu_baseline(args, scn, env, oracle, frame=args.warmup + k)
        tot_t += dt
        tot_r += rays
    val = tot_r / tot_t / 1e6
    cb["value"] = val
    line = {"impl": "reference", "metric": CONFIG_SCENES[args.config][1], "value": val, "unit": "Mray/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / max(args.steps, 1), "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args, scn, 1),
            "cpu_baseline": cb, "e2e": {"value": val, "unit": "Mray/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "note": "each step = the sample band of one 1080p frame on the host cores; Mray/s is size-independent"}
    emit(line)


def traversal_counts(args, scn, env, device):
    """Per-ray node / triangle averages on the SAME BVH and the same frame, from the counter build of the library."""
    from vk_gltf_renderer_b200.renderer import PathTracer, Resources
    res = Resources(scene=scn, hdr_rgb=env, camera=scn.camera, size=(args.width, args.height))
    pt = PathTracer(device, count_traversal=True)
    pt.ptMaxDepth = args.depth
    pt.onAttach(res)
    res.frameCount = 0
    pt.onRender(None, res)
    st = pt.stats()
    pt.onDetach()
    rays = st["closestRays"] + st["shadowRays"]
    return st["nodesVisited"] / max(rays, 1), st["trisTested"] / max(rays, 1), st


def main():
    args = parse()
    # the contract is ONE JSON line on stdout: libraries (NCCL banner, torch warnings) that print to fd 1 are sent to stderr
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = sys.stderr

    def emit(obj):
        real_stdout.write(json.dumps(obj) + "\n")
        real_stdout.flush()
    if args.impl == "reference":
        run_reference(args, emit)
        return
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        args.gpus = world
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from vk_gltf_renderer_b200.renderer import PathTracer, Resources
    scn, env = build_workload(args)
    W, H = args.width, args.height
    from vk_gltf_renderer_b200 import tiling
    band = tiling.interleave_band(H, world)
    if band:
        # interleaved bands of `band` rows: every rank gets a fair mix of cheap (sky) and expensive (atrium) rows
        rows_per = rows = H // world
        y0 = 0
        tile_spec = ("interleave", band, world, rank)
    else:
        rows_per = tiling.strip_rows(H, world)
        y0, rows = tiling.partition_rows(H, world, rank)
        tile_spec = (y0, rows)
    res = Resources(scene=scn, hdr_rgb=env, camera=scn.camera, size=(W, H), tile=tile_spec)
    pt = PathTracer(local)
    pt.ptMaxDepth = args.depth
    pt.onAttach(res)
    # Frames in flight hide the latency-bound tails of a frame behind the wide bounces of the next ones; frame batching
    # (b200pt_set_frame_batch) runs consecutive frames as ONE wavefront, which makes the tails of a frame wider and divides the
    # launches per frame.  At N > 1 a rank's tile is 1/N of the frame, so the batch grows with N and every kernel keeps the size it
    # has on one GPU (round 1, one frame per launch chain: 0.61 efficiency at N = 8).
    lanes = 4
    # measured at N = 1 (r02m, frames in flight 4): batch 1 -> 821 (r02g), 4 -> 926, 6 -> 949, 8 -> 947 Mray/s.  The batch grows with N so
    # that a rank's wavefront stays as large as on one GPU, but never beyond half the timed steps (two wavefronts overlap their tails)
    # (r02y / r02z, --steps 20: two equal wavefronts of 10 frames 987 / 994 Mray/s against 8 + 8 + 4 at 981 / 988)
    batch = max(1, min(8 * world if world > 1 else 16, 64, (args.steps + 1) // 2))
    if os.environ.get("B200PT_FRAMES_IN_FLIGHT"):
        lanes = int(os.environ["B200PT_FRAMES_IN_FLIGHT"])
    if os.environ.get("B200PT_FRAME_BATCH"):
        batch = int(os.environ["B200PT_FRAME_BATCH"])
    pt.set_frames_in_flight(lanes)
    pt.set_frame_batch(batch)
    stream = torch.cuda.ExternalStream(pt.stream(), device=local)
    tile = torch.zeros((rows_per, W, 4), dtype=torch.float32, device="cuda")
    pt.set_accum_device(tile.data_ptr(), rows * W * 4)
    full = torch.empty((world * rows_per, W, 4), dtype=torch.float32, device="cuda") if world > 1 else None
    RING = 8  # read-back ring (one pinned image per frame / batch in flight)
    pinned = [torch.empty((H if world > 1 else rows, W, 4), dtype=torch.float32).pin_memory() for _ in range(RING if (world == 1 or rank == 0) else 0)]

    frame = [-1]
    image = [None]
    pending = [0]

    def finish_batch():
        """the frames submitted since the last call are enqueued (flush) and, at N > 1, the tiles all-gathered into the image"""
        if pending[0] == 0:
            return
        pending[0] = 0
        pt.flush()
        if world > 1:
            with torch.cuda.stream(stream):
                dist.all_gather_into_tensor(full, tile)
                image[0] = tiling.deinterleave(full, H, world, band) if band else full  # rank-major bands -> image order (device copy)

    def step():
        frame[0] += 1
        res.frameCount = frame[0]
        pt.onRender(None, res)
        pending[0] += 1
        if pending[0] >= batch:
            finish_batch()

    def barrier():
        torch.cuda.synchronize()
        pt.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(n, fn):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(n):
            fn()
        finish_batch()  # a partial last batch belongs to the timed steps
        e1.record(stream)
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    def rays_now():
        st = pt.stats()
        r = torch.tensor([st["closestRays"] + st["shadowRays"], st["closestRays"], st["shadowRays"], st["shadedHits"], st["kernelLaunches"]],
                         dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(r)
        return r.cpu().numpy()

    def dump_outputs():
        """rank 0 writes the accumulation image after the last timed step (at N > 1 the gathered full frame)"""
        if not args.dump_outputs or rank != 0:
            return
        img = (image[0][:H] if world > 1 else tile[:rows]).cpu().numpy()
        stride = max(1, math.ceil(img.nbytes / DUMP_BYTES))  # a fixed row sample keeps 4K frames under the limit
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "accum.npy"), np.ascontiguousarray(img[::stride]))

    # ---- warm-up ----
    if args.profile_only:
        for _ in range(args.warmup + args.steps):
            step()
        finish_batch()
        barrier()
        dump_outputs()
        return
    for _ in range(max(args.warmup, 3)):
        step()
    finish_batch()
    # ---- pass A: device-timed throughput (headline `value`) ----
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    pt.reset_stats()
    ms = timed(args.steps, step)
    cl = clocks.stop() if rank == 0 else None
    dump_outputs()
    r = rays_now()
    rays_total, launches = r[0], int(r[4])
    value = rays_total / (ms * 1e-3) / 1e6
    spp_per_s = args.steps / (ms * 1e-3)

    # ---- pass B: same steps with per-launch CUDA events -> stage shares + roofline ----
    pt.set_profiling(True)
    pt.reset_stats()
    timed(args.steps, step)
    stB = pt.stats()
    pt.set_profiling(False)

    # ---- pass C: end to end through the public API with host buffers ----
    # every step: submit the frame (444 B of frame constants go host->device as kernel arguments), then read the
    # step's image back into pinned host memory.  The read-back is ring-buffered like the reference's staging
    # ring: the copy of frame f is enqueued behind its accumulate, and the host consumes frame f-depth (waits for
    # its copy, touches the pixels) while the newer frames render.  The last frames are consumed before the clock stops.
    checks = []
    depth = min(lanes, RING) - 1  # the host consumes image k-depth while the newer ones render

    # After every batch the image is read back into pinned host memory (N > 1: rank 0 reads the GATHERED full-resolution image,
    # the frame the metric describes; the other ranks only take part in the gather).  A batch's frames complete together, so the
    # image after an intermediate frame never exists: one read per batch is every result there is.  (The reference's headless run
    # reads its image back once, at the end.)  The per-frame variant is measured separately below.
    copies = []
    src_image = (lambda: image[0]) if world > 1 else (lambda: tile)

    def consume(k):
        copies[k].synchronize()
        checks.append(float(pinned[k % RING][0, 0, 3]))

    def read_back():
        j = len(copies)
        with torch.cuda.stream(stream):
            pinned[j % RING].copy_(src_image(), non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(stream)
        copies.append(ev)
        if j >= depth:
            consume(j - depth)

    def step_e2e(k):
        step()
        if pending[0] == 0 and rank == 0:  # a batch just completed (and was gathered)
            read_back()
    pt.reset_stats()
    barrier()
    t0 = time.perf_counter()
    for k in range(args.steps):
        step_e2e(k)
    if pending[0]:
        finish_batch()
        if rank == 0:
            read_back()
    if rank == 0:
        for j in range(max(len(copies) - depth, 0), len(copies)):
            consume(j)
    n_reads = len(copies)
    barrier()
    dt = torch.tensor([time.perf_counter() - t0], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    re = rays_now()
    e2e_val = re[0] / float(dt.item()) / 1e6
    # the same with the image read back after EVERY frame (N = 1 only): each read flushes the pending batch, so this is the
    # unbatched renderer end to end
    e2e_per_frame = None
    if world == 1:
        pt.reset_stats()
        barrier()
        t0 = time.perf_counter()
        for k in range(args.steps):
            step()
            pt.read_accum_async(pinned[k % RING].data_ptr(), pinned[k % RING].numel(), k % RING)
            pending[0] = 0
            if k >= depth:
                pt.wait_read((k - depth) % RING)
        for k in range(max(args.steps - depth, 0), args.steps):
            pt.wait_read(k % RING)
        barrier()
        e2e_per_frame = rays_now()[0] / (time.perf_counter() - t0) / 1e6

    # ---- pass D: the same steps on the same scene carrying opacity micromaps (an asset with EXT_mesh_opacity_micromap: the walk
    # resolves OPAQUE / TRANSPARENT micro-triangles itself, csrc/omm.cuh).  Reported beside the headline, never as it: the stand-in
    # asset, like the Sponza it stands for, has no micromaps.
    omm_extra = None
    if args.omm == 0 and not args.no_omm_pass and args.config in (3, 5):
        from vk_gltf_renderer_b200 import omm as ommod
        t_b = time.perf_counter()
        st_omm = ommod.bake_opacity_micromaps(scn, level=5)
        bake_s = time.perf_counter() - t_b
        if st_omm["triangles"]:
            barrier()
            pt.onSceneInvalidated(res)  # SceneOmm::create + the tree build that consumes it
            for _ in range(max(args.warmup, 3)):
                step()
            finish_batch()
            pt.reset_stats()
            ms_o = timed(args.steps, step)
            r_o = rays_now()
            omm_extra = {"value": r_o[0] / (ms_o * 1e-3) / 1e6, "unit": "Mray/s", "ms_per_step": ms_o / args.steps, "subdivision_level": 5,
                         "alpha_triangles": st_omm["triangles"], "unknown_fraction": st_omm["unknown"] / max(st_omm["micro"], 1), "bake_s": bake_s,
                         "note": "same scene, camera, steps and batching with opacity micromaps baked from the MASK texture (vk_gltf_renderer_b200/omm.py, "
                                 "untimed like the BVH build); rays per frame are the same, the any-hit work is what shrinks; parity: tests/test_gpu_omm.py"}
        scn.micromaps, scn.prim_omms, scn._keep = [], [], []  # the counters and the CPU baseline below see the asset as it is

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline model (rank 0) ----
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    nn = nt = None
    counts_note = "skipped"
    if world == 1:
        nn, nt, stc = traversal_counts(args, scn, env, local)
        counts_note = "frame 0, counter build of the same library: %.2f nodes/ray, %.2f tris/ray" % (nn, nt)
    stages = {}
    tot_ms = max(stB["msTotal"], 1e-9)
    closest_b = shadow_b = None
    if nn is not None:
        closest_b = 32 + 24 + nn * NODE_BYTES + nt * TRI_BYTES
        shadow_b = 32 + 16 + nn * NODE_BYTES + nt * TRI_BYTES
    shade_b = 1100.0  # SURVEY.md §8d: ~1.0-1.2 KB per shaded hit
    # one entry per kernel kind; the tree walks carry the algorithmic-bytes model (node + triangle records a ray touches),
    # the dense kernels are listed with their time share only
    for name, ms_k, n_l, units, per in (("k_trace", stB["msTraceClosest"], stB["launchesTraceClosest"], stB["closestRays"], closest_b),
                                        ("k_shade", stB["msShade"], stB["launchesShade"], stB["shadedHits"], shade_b),
                                        ("k_shadow", stB["msTraceShadow"], stB["launchesTraceShadow"], stB["shadowRays"], shadow_b),
                                        ("k_alpha", stB["msAnyHit"], stB["launchesAnyHit"], 0, None),
                                        ("k_resolve", stB["msResolve"], stB["launchesResolve"], 0, None)):
        ach = (units * per / (ms_k * 1e-3) / 1e9) if (per and ms_k > 0) else None
        stages[name] = {"share": ms_k / tot_ms, "ms_per_launch": ms_k / max(n_l, 1), "launches": int(n_l), "units": int(units),
                        "bytes_per_unit": per, "achieved_GBps": ach}
    dom = max(stages, key=lambda k: stages[k]["share"])
    # measured DRAM traffic of the dominant kernel: one `ncu --set full` capture, per launch (profiles/ncu_traffic.json)
    try:
        ncu_traffic = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    except Exception:
        ncu_traffic = {}
    tr = ncu_traffic.get(dom) if (args.config == 3 and world == 1) else None  # the capture is of the default workload
    if tr:
        tr = dict(tr, note="dram__bytes_read.sum + dram__bytes_write.sum of ONE launch from the committed `ncu --set full` capture named in "
                           "`source` (taken with this build under the profiler, not during this run)")
    roof = {"kernel": dom, "bound": "hbm", "achieved": stages[dom]["achieved_GBps"], "peak": peak_gbs, "unit": "GB/s",
            "frac": (stages[dom]["achieved_GBps"] / peak_gbs) if stages[dom]["achieved_GBps"] else None,
            "traffic": tr["bytes"] if tr else None, "traffic_detail": tr,
            "peak_source": peak_src, "model": "algorithmic bytes/unit x units / CUDA-event kernel time (pass B); " + counts_note,
            "stages": stages}

    cb = None
    if not args.no_cpu_baseline and world == 1:
        _, cb, _, _ = cpu_baseline(args, scn, env)

    line = {"metric": CONFIG_SCENES[args.config][1], "value": value, "unit": "Mray/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(args, scn, world), "spp_per_s": spp_per_s,
            "throughput_MSps": W * H * spp_per_s / 1e6, "rays_per_sample": rays_total / (args.steps * W * H),
            "clocks": cl, "e2e": {"value": e2e_val, "unit": "Mray/s", "h2d_bytes_per_step": 396 + 48,
                                  "d2h_bytes_per_step": (H * W * 16 * n_reads) // max(args.steps, 1),
                                  "d2h_note": "the image is read back once per batch of frame_batch frames (rank 0 reads the gathered full image); "
                                              "per_frame_readback_value = the same metric with a read after every frame (N = 1)",
                                  "per_frame_readback_value": e2e_per_frame,
                                  "ms_per_step": 1e3 * float(dt.item()) / args.steps},
            "frames_in_flight": lanes, "frame_batch": batch,
            "gpu_launches": launches, "roofline": roof, "cpu_baseline": cb, "with_opacity_micromaps": omm_extra}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
