#!/usr/bin/env python
"""bench.py — one "step" = one frame of the hot path (prepass rays + light passes + denoise + tone mapping).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config cornell_1080p] [--impl ours|reference] [--dump-outputs DIR]

N = 1: the workload is BASELINE.json configs[1] — cornell 1920x1080, 2 bounces, ReSTIR temporal + spatial (emissive
and indirect), denoise on — unless --config says otherwise.  N > 1 (launched by torchrun, one rank per GPU): the frame is
split in N equal screen tiles (a columns x rows grid, SURVEY.md 8(e)); every rank renders its tile + ghost pixels with no
data-path exchange, then ONE NCCL all-gather collects the tone-mapped tiles on every rank (tile-major: [rank][row][col]) ("scaling": "strong" — total work is fixed).

Timing: W warm-up frames, then exactly K frames bracketed by barrier + torch.cuda.synchronize(), CUDA events on the
context's stream (which is torch's current stream), MAX over ranks.  Frames continue the temporal sequence
(frame numbers W+1 .. W+K), so validation frames (every 3rd / 5th) are inside the timed region.  The per-frame working
set (~880 B/px of planes = 1.8 GB at 1080p) is far larger than the 126 MB L2, so no explicit flush is needed.

value      Mrays/s, device-resident: rays = traverse_top calls + stand-alone traverse_bottom calls of the light passes
           (SURVEY.md 8(d)), counted exactly by replaying the same frames with the counting kernel variants AFTER the timed
           region (counters are compiled out of the timed kernels); primary (G-buffer) rays are reported separately.
e2e        same metric through the public plugin API with host buffers: HikariPlugin.run_frame(settings, view, lights)
           (host structs -> kernel parameters) + read-back of the tone-mapped tile into pinned host memory every frame,
           pipelined like a presentation loop: hk_readback_async copies frame n on the context's copy stream while frame
           n + 1 renders; the host waits for (and so observes) every frame's image, the last one inside the timed region.
roofline   dominant kernel (largest share of the frame): algorithmic bytes/pixel (SURVEY.md 8(d)) x pixels / its mean
           CUDA-event time, against MEASURED_PEAKS.json hbm_gbs.
cpu_baseline / --impl reference: the oracle (CPU restatement of the reference's WGSL; the reference itself is Rust + wgpu
           and cannot be built offline) on the host cores.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# algorithmic bytes per render pixel (SURVEY.md 8(d)): unique compulsory traffic of each reference pass
BYTES_PER_PIXEL = {"gbuffer": 52 + 52, "direct": 184, "emissive": 184, "emissive_spatial": 244, "indirect": 184,
                   "indirect_spatial": 244, "demodulation": 32, "denoise_0": 56, "denoise_1": 56, "denoise_2": 56,
                   "denoise_3": 56 + 8, "tone_mapping": 32}
PER_SIGNAL = {"demodulation", "denoise_0", "denoise_1", "denoise_2", "denoise_3"}   # x signals (fused over signals here)


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons (B200_PROFILING.md).  Started BEFORE the warm-up frames and left running through both
    timed arms: spawning nvidia-smi takes hundreds of milliseconds of driver initialisation, which stalls kernel launches of every
    process on the box — round 1 started it right before a 14 ms timed region at 8 GPUs and measured its own start-up.  Samples carry
    host timestamps; `window(t0, t1)` summarises the ones taken under load."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "25",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
            t0 = time.time()
            while not self.lines and time.time() - t0 < 5.0:      # first sample printed: start-up is over
                time.sleep(0.05)
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self):
        if not self.proc:
            return
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()

    def window(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm, mx, reasons = [], [], set()
        for t, l in self.lines:
            if t < t0 or t > t1 + 0.11:
                continue
            p = [x.strip() for x in l.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); mx.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm),
                "window": "warm-up + both timed arms (sampler started before the warm-up; 25 ms period)"}


GHOST = 36   # rows / columns a tile renders beyond its own rectangle (bevy_hikari_b200/csrc/context.cu GHOST_TEMPORAL)


def tile_grid(width, height, world):
    """(columns, rows) of the tile grid for `world` GPUs: equal tiles (the all-gather needs equal contributions), the
    factorisation with the most columns among those within 5 % of the least rendered area (incl. ghost pixels): vertical
    strips share sky / ground evenly, row bands do not."""
    cands = []
    for cx in range(1, world + 1):
        if world % cx:
            continue
        cy = world // cx
        if width % cx or height % cy:
            continue
        tw, th = width // cx, height // cy
        area = 0
        for j in range(cy):
            for i in range(cx):
                w = min(width, (i + 1) * tw + GHOST) - max(0, i * tw - GHOST)
                h = min(height, (j + 1) * th + GHOST) - max(0, j * th - GHOST)
                area += w * h
        cands.append((area, cx, cy))
    assert cands, "image size must be divisible by a factorisation of the number of GPUs"
    least = min(a for a, _, _ in cands)
    area, cx, cy = max((c for c in cands if c[0] <= 1.05 * least), key=lambda c: c[1])   # most columns within 5 % of the least area
    return cx, cy


def tile(width, height, rank, world):
    """(x0, x1, y0, y1) owned by `rank`; ranks run left to right, then top to bottom."""
    cx, cy = tile_grid(width, height, world)
    tw, th = width // cx, height // cy
    i, j = rank % cx, rank // cx
    return i * tw, (i + 1) * tw, j * th, (j + 1) * th


def balanced_cuts(cost, n, align=8):
    """cut positions (n + 1 of them, multiples of `align` except the last) splitting `cost` (per line) into n parts of
    nearly equal sum"""
    L = len(cost)
    pre = np.concatenate([[0.0], np.cumsum(cost)])
    cuts = [0]
    for k in range(1, n):
        pos = int(np.searchsorted(pre, pre[-1] * k / n))
        pos = int(round(pos / align)) * align
        pos = max(cuts[-1] + align, min(pos, L - align * (n - k)))
        cuts.append(pos)
    cuts.append(L)
    return cuts


def plan_tiles(width, height, world, coverage=None, background_weight=0.15, ghost=GHOST):
    """One (x0, x1, y0, y1) per rank.  Without a coverage map: the equal grid of tile().  With one (H' x W' booleans from
    a low-resolution primary-ray pass, identical on every rank): every factorisation cx x cy of `world` is tried — vertical strips,
    horizontal strips and 2-D grids — with cuts that equalise the estimated cost along each axis (covered pixels +
    `background_weight` per pixel), and the plan whose most expensive tile INCLUDING ITS GHOST RING is cheapest wins.  A 4 x 2 grid at
    8 GPUs renders 30 % ghost pixels where 8 strips of a 1080p frame render 56 %.  Ranks run left to right, then top to bottom."""
    if world == 1:
        return [(0, width, 0, height)]
    if coverage is None:
        return [tile(width, height, r, world) for r in range(world)]
    cov = np.asarray(coverage, np.float64)
    ry, rx = int(round(height / cov.shape[0])), int(round(width / cov.shape[1]))
    cost = np.repeat(np.repeat(cov + background_weight, ry, axis=0), rx, axis=1)[:height, :width] / (ry * rx)
    if cost.shape != (height, width):
        cost = np.pad(cost, ((0, height - cost.shape[0]), (0, width - cost.shape[1])), mode="edge")
    pre = np.zeros((height + 1, width + 1))
    pre[1:, 1:] = cost.cumsum(axis=0).cumsum(axis=1)

    def rect(x0, x1, y0, y1):
        return pre[y1, x1] - pre[y0, x1] - pre[y1, x0] + pre[y0, x0]

    best = None
    for cx in range(1, world + 1):
        if world % cx:
            continue
        cy = world // cx
        if width < cx * 2 * ghost or height < cy * 2 * ghost:
            continue
        xcuts = balanced_cuts(cost.sum(axis=0), cx) if cx > 1 else [0, width]
        ycuts = balanced_cuts(cost.sum(axis=1), cy) if cy > 1 else [0, height]
        tiles = [(xcuts[i], xcuts[i + 1], ycuts[j], ycuts[j + 1]) for j in range(cy) for i in range(cx)]
        worst = max(rect(max(0, x0 - ghost), min(width, x1 + ghost), max(0, y0 - ghost), min(height, y1 + ghost)) for x0, x1, y0, y1 in tiles)
        if best is None or worst < best[0] * 0.999:
            best = (worst, tiles)
    if best is None:
        return [tile(width, height, r, world) for r in range(world)]
    return best[1]


ASSET_OF = {"cornell": "cornell.glb", "city": "Low Poly/Big House{, 2, 3}.glb + Earth/earth_daymap.jpg",
            "town": "scene.gltf + Earth/earth_daymap.jpg, textures box-filtered to <= 256 px", "terrain": "procedural stress scene",
            "minimal": "bevy shapes", "simple": "bevy shapes", "samplers": "procedural"}


def make_bench(config):
    from bevy_hikari_b200 import plugin, scenes
    cfg = scenes.CONFIGS[config]
    scene = scenes.SCENE_BUILDERS[cfg["scene"]]()
    world = scene.populate(plugin.World())
    W, H = cfg["width"], cfg["height"]
    view, pview, lights = scene.view_inputs(W, H)
    settings = scenes.config_settings(config)
    return cfg, scene, world, W, H, view, pview, lights, settings


def config_json(config, cfg, settings, world_size, gather="peer"):
    return {"workload": f"{config}: {cfg['scene']} {cfg['width']}x{cfg['height']}, {settings.indirect_bounces} bounces, "
                        f"temporal+{'emissive+' if settings.emissive_spatial_reuse else ''}"
                        f"{'indirect ' if settings.indirect_spatial_reuse else ''}spatial ReSTIR, denoise {'on' if settings.denoise else 'off'}",
            "scene": cfg["scene"], "width": cfg["width"], "height": cfg["height"], "indirect_bounces": int(settings.indirect_bounces),
            "emissive_spatial_reuse": int(settings.emissive_spatial_reuse), "indirect_spatial_reuse": int(settings.indirect_spatial_reuse),
            "denoise": int(settings.denoise), "upscale": "SmaaTu4x{ratio:1.0}", "taa": "None",
            "parallelism": (f"{world_size} screen tiles (+{GHOST} ghost px each side, cuts balanced on a coverage probe unless "
                            "--equal-tiles), " + ("tiles stored by the tone-map kernel into rank 0's frame over NVLink (CUDA IPC) + a 4-byte "
                                                 "all-reduce as the frame barrier" if gather == "peer" else
                                                 "one all-gather of the tone-mapped tiles")) if world_size > 1 else "single GPU",
            "l2": ((f"per-frame working set ({876 * cfg['width'] * cfg['height'] / 1e6:.0f} MB of per-pixel planes) exceeds the 126 MB L2; no explicit flush")
                   if 876 * cfg["width"] * cfg["height"] > 2 * 126e6 else
                   (f"per-frame working set ({876 * cfg['width'] * cfg['height'] / 1e6:.0f} MB) fits L2 and is NOT flushed between frames: "
                    "consecutive frames of a frame loop are L2-warm by nature; not a roofline configuration"))}


# ================================================================================================== ours
def run_ours(args):
    import torch
    import torch.distributed as dist
    from bevy_hikari_b200 import layout as L
    from bevy_hikari_b200 import plugin

    rank = int(os.environ.get("RANK", "0"))
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world_size > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    assert world_size == args.gpus or world_size == 1, "launch with torchrun --nproc-per-node N for --gpus N"

    cfg, scene, world, W, H, view, pview, lights, settings = make_bench(args.config)
    tiles = None
    if world_size > 1 and not args.equal_tiles:
        # coverage map from a quarter-resolution primary-ray pass on this rank's own GPU (bit-identical on every rank,
        # so every rank derives the same plan without communicating)
        cw, ch = max(W // 4, 1), max(H // 4, 1)
        probe = plugin.HikariPlugin(cw, ch, cuda_device=local_rank)
        probe.upload_scene(world)
        pv, ppv, pl = scene.view_inputs(cw, ch)
        probe.prepass(plugin.make_frame_inputs(settings, 1, pv, ppv, pl))
        coverage = probe.readback(L.OUT_GBUFFER_INSTANCE_MATERIAL)[..., 0] > 0
        probe.close()
        tiles = plan_tiles(W, H, world_size, coverage)
    else:
        tiles = plan_tiles(W, H, world_size)
    x0, x1, r0, r1 = tiles[rank]
    # a dedicated non-default stream, made torch's current stream so that torch.cuda.Event, NCCL and the context's
    # kernels are all ordered on the same stream (the legacy default stream has handle 0 = "create your own" in the C ABI)
    stream = torch.cuda.Stream(device=local_rank)
    torch.cuda.set_stream(stream)
    dev = plugin.HikariPlugin(W, H, cuda_device=local_rank, row_begin=r0, row_end=r1, cuda_stream=stream.cuda_stream,
                              col_begin=x0, col_end=x1)
    if world_size > 1 and args.halo_margin is not None:
        dev.set_motion_margin(args.halo_margin)      # re-allocates the tile with 36 + margin ghost pixels (before any pointer is taken)
    dev.upload_scene(world)

    # the context's tone-mapped band as a torch tensor (zero copy) for the all-gather
    ptr, nbytes = dev.output_device_pointer()

    class _Ext:  # __cuda_array_interface__ view of the context-owned buffer
        __cuda_array_interface__ = {"shape": (nbytes // 2,), "typestr": "<f2", "data": (ptr, False), "version": 3}
    tile_t = torch.as_tensor(_Ext(), device=f"cuda:{local_rank}")
    # tiles may differ in size (balanced cuts): every rank contributes a buffer padded to the largest tile
    max_elems = max((t[1] - t[0]) * (t[3] - t[2]) for t in tiles) * 4
    send_buf = torch.zeros(max_elems, dtype=torch.float16, device=tile_t.device) if world_size > 1 else None
    frame_buf = torch.empty(world_size * max_elems, dtype=torch.float16, device=tile_t.device) if world_size > 1 else None

    # Frame assembly (N > 1).  Default: rank 0 owns two full-frame buffers (double-buffered); every rank maps them through
    # CUDA IPC and its last kernel stores the tile's pixels straight into the frame over NVLink (hk_set_frame_target) —
    # the store is the transfer; the only collective is a 4-byte all-reduce that tells rank 0 that every tile has landed.
    # --gather nccl keeps the earlier form (copy + all_gather_into_tensor of padded tiles) for comparison.
    frame_targets = None
    landed = torch.zeros(1, dtype=torch.int32, device=tile_t.device) if world_size > 1 else None
    if world_size > 1 and args.gather == "peer":
        handles = [None, None]
        if rank == 0:
            own = [dev.frame_alloc(), dev.frame_alloc()]
            frame_targets = [own[0][0], own[1][0]]
            handles = [own[0][1], own[1][1]]
        dist.broadcast_object_list(handles, src=0)
        ok = torch.ones(1, dtype=torch.int32, device=tile_t.device)
        if rank != 0:
            try:
                frame_targets = [dev.frame_open(handles[0]), dev.frame_open(handles[1])]
            except Exception as e:      # no CUDA IPC between the ranks on this box: every rank falls back together
                print(f"bench.py: rank {rank}: hk_frame_open failed ({e}); falling back to --gather nccl", file=sys.stderr)
                ok.zero_()
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            frame_targets = None
            args.gather = "nccl"
    # Exact tiling under camera motion (--halo-margin M, off by default; the benchmark camera is static, so this measures the
    # cost of the exchange, the exactness is tests/test_gpu_zz_halo.py): every rank maps every other rank's reservoir planes
    # through CUDA IPC once; after each frame, between two frame barriers, it pulls the part of its ghost ring each owns.
    halo_peers = []
    if world_size > 1 and args.halo_margin is not None:
        descriptors = [None] * world_size
        dist.all_gather_object(descriptors, dev.halo_export())
        halo_peers = [dev.halo_import(d) for r, d in enumerate(descriptors) if r != rank]
    frame_no = [0]

    def begin_frame():
        if frame_targets:
            dev.set_frame_target(frame_targets[frame_no[0] & 1], W)
        frame_no[0] += 1

    def gather_frame():
        if frame_targets:
            dist.all_reduce(landed)          # stream-ordered behind this rank's tone-map stores: "all tiles have landed"
        else:
            send_buf[:tile_t.numel()].copy_(tile_t)
            dist.all_gather_into_tensor(frame_buf, send_buf)
        if halo_peers:                       # every rank has finished the frame (collective above): refresh the ghost ring
            for peer in halo_peers:
                dev.halo_pull_peer(peer)
            dist.all_reduce(landed)          # nobody overwrites reservoirs a neighbour is still reading
    pinned = torch.empty(nbytes, dtype=torch.uint8).pin_memory()

    def barrier():
        if world_size > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(x):
        if world_size == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=tile_t.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def reduce_sum(vals):
        if world_size == 1:
            return vals
        t = torch.tensor(vals, dtype=torch.float64, device=tile_t.device)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [float(v) for v in t.tolist()]

    W_, K = args.warmup, args.steps
    dev.set_temporal_upscalers(False)        # SURVEY 8(d): the benchmarked path ends at the tone-mapped image (SmaaTu4x{ratio 1}, Taa::None)

    # --moving-camera: the camera translates a little every frame (about a pixel of image motion), so that temporal reprojection
    # crosses tile borders — the case the reservoir-halo exchange (--halo-margin) exists for.  Default: the static benchmark camera.
    views, pviews = [view] * (W_ + K + 1), [pview] * (W_ + K + 1)
    if args.moving_camera:
        from bevy_hikari_b200 import camera as cam
        step = (0.003, 0.001, -0.002)

        def view_at(f):
            eye = tuple(e + d * (f - 1) for e, d in zip(scene.eye, step))
            tgt = tuple(t + d * (f - 1) for t, d in zip(scene.target, step))
            return cam.make_view(cam.look_at(eye, tgt), cam.perspective_infinite_reverse_rh(scene.fov, W / H, scene.near), W, H)
        views = [view_at(f) for f in range(1, W_ + K + 2)]
        pviews = [cam.make_previous_view(view_at(max(f - 1, 1))) for f in range(1, W_ + K + 2)]

    def frame_inputs(n):
        return plugin.make_frame_inputs(settings, n, views[n - 1], pviews[n - 1], lights)

    inputs = [frame_inputs(n) for n in range(1, W_ + K + 1)]
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()                      # long before any timed region (see ClockSampler)
    barrier()
    t_load_begin = time.time()

    # ------------------------------------------------ replay 1: per-kernel times (every kernel bracketed with events, one sync per
    # frame) -> which kernel dominates; outside every timed region
    dev.set_profiling(False, True)
    dev.set_profiling_kernel(-1)
    dev.reset_temporal_state()
    kernel_ms = np.zeros(len(L.KERNEL_NAMES))
    launches = 0
    for n in range(W_ + K):
        dev.render_frame(inputs[n])
        if n >= W_:
            st = dev.stats()
            kernel_ms += np.array(st.ms_kernel[:len(L.KERNEL_NAMES)])
            launches += st.kernel_launches
    kernel_ms /= K
    launches_per_frame = launches // K + (1 if world_size > 1 else 0)
    dominant = int(np.argmax(kernel_ms))

    # ------------------------------------------------ replay 2: exact ray counts of the timed frames (counting kernel variants)
    dev.reset_temporal_state()
    dev.set_profiling(True, False)
    rays = np.zeros(3)
    for n in range(W_ + K):
        dev.render_frame(inputs[n])
        if n >= W_:
            st = dev.stats()
            rays += np.array([st.primary_rays, st.tlas_rays, st.blas_rays], dtype=np.float64)
    rays = np.array(reduce_sum(list(rays)))
    light_rays = rays[1] + rays[2]

    # ---------------------------------------------------------------- device-resident arm ("value")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    frame_events = [torch.cuda.Event(enable_timing=True) for _ in range(K)]

    def measure_value():
        """W warm-up frames, then exactly K frames between barrier + synchronize; inside the timed region the only event records
        are one per frame (per-frame times) and, at N = 1, the two that bracket the dominant kernel (hk_set_profiling_kernel)."""
        dev.reset_temporal_state()
        dev.set_profiling(False, False)
        dev.set_profiling_kernel(dominant if world_size == 1 else -1)
        frame_no[0] = 0
        for n in range(W_):
            begin_frame()
            dev.render_frame(inputs[n])
            if world_size > 1:
                gather_frame()
        if world_size == 1:
            dev.set_profiling_kernel(dominant)   # restart the ring: only timed frames are averaged
        barrier()
        e0.record(stream)
        for n in range(W_, W_ + K):
            begin_frame()
            dev.render_frame(inputs[n])
            if world_size > 1:
                gather_frame()
            frame_events[n - W_].record(stream)
        e1.record(stream)
        barrier()
        per_frame = [e0.elapsed_time(frame_events[0])] + [frame_events[i - 1].elapsed_time(frame_events[i]) for i in range(1, K)]
        dom_live = None
        if world_size == 1:
            st = dev.stats()
            dom_live = float(st.ms_kernel[dominant]) if st.timed_frames else None
            dev.set_profiling_kernel(-1)
        return reduce_max(e0.elapsed_time(e1)), per_frame, dom_live

    # ---------------------------------------------------------------- end-to-end arm ("e2e")
    h2d = ctypes.sizeof(L.FrameInputs)
    # Presentation-loop form: frame n's tile is copied to pinned host memory on the context's copy stream while frame
    # n + 1 renders (hk_readback_async); the host sees every frame's result, one frame later.  Two pinned buffers alternate.
    pinned2 = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    host_bufs = [pinned.data_ptr(), pinned2.data_ptr()]
    d2h_bytes = nbytes
    if frame_targets:
        # N > 1: the tiles land in rank 0's frame over NVLink; rank 0 reads the ASSEMBLED frame back to pinned host memory
        # on a copy stream while the next frame renders.  Buffer (n & 1) is rewritten by frame n + 2: rank 0 orders its
        # frame barrier n + 1 behind copy n, so no rank can store frame n + 2 before that copy has finished.
        frame_bytes = W * H * 8
        d2h_bytes = frame_bytes if rank == 0 else 0
        copy_stream = torch.cuda.Stream(device=local_rank)
        copied = torch.cuda.Event()
        if rank == 0:
            class _Frame:
                def __init__(self, ptr):
                    self.__cuda_array_interface__ = {"shape": (frame_bytes,), "typestr": "|u1", "data": (ptr, False), "version": 3}
            frame_views = [torch.as_tensor(_Frame(p), device=f"cuda:{local_rank}") for p in frame_targets]
            host_frames = [torch.empty(frame_bytes, dtype=torch.uint8, pin_memory=True) for _ in range(2)]

        def e2e_step(n, first, i):
            begin_frame()
            dev.run_frame(settings, views[i], pviews[i], lights)
            if rank == 0 and not first:
                stream.wait_event(copied)            # frame barrier n is ordered behind copy n - 1
            gather_frame()
            if rank == 0:
                ready = torch.cuda.Event()
                ready.record(stream)
                if not first:
                    copied.synchronize()             # the host observes frame n - 1
                copy_stream.wait_event(ready)
                with torch.cuda.stream(copy_stream):
                    host_frames[n & 1].copy_(frame_views[(frame_no[0] - 1) & 1], non_blocking=True)
                    copied.record(copy_stream)

        def e2e_finish():
            if rank == 0:
                copied.synchronize()
    else:
        def e2e_step(n, first, i):
            dev.run_frame(settings, views[i], pviews[i], lights)              # host structs -> kernel parameters
            dev.readback_wait()                                               # frame n - 1 has landed in host memory
            dev.readback_async(L.OUT_TONE_MAPPED, host_bufs[n & 1], nbytes)   # D2H of this frame's tile, overlapping the next frame
            if world_size > 1:
                gather_frame()

        def e2e_finish():
            dev.readback_wait()                                               # the last frame's result too

    def measure_e2e():
        dev.set_profiling(False, False)
        dev.set_profiling_kernel(-1)
        dev.reset_temporal_state()
        dev.frame_counter = 0
        frame_no[0] = 0
        for n in range(W_):
            e2e_step(n, n == 0, n)
        e2e_finish()
        barrier()
        t0 = time.perf_counter()
        e0.record(stream)
        for n in range(K):
            e2e_step(n, n == 0, W_ + n)
        e2e_finish()
        e1.record(stream)
        barrier()
        return reduce_max(max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3))

    # The two arms time the same K frames; the end-to-end one adds the read-back, which overlaps the next frame, so they must agree
    # closely.  A disagreement beyond 15 % means one of them measured something else (round 1, 8 GPUs: 5x) — measure again, once,
    # and say so.
    attempts = []
    for attempt in range(2):
        ms_total, per_frame, dom_live = measure_value()
        e2e_ms = measure_e2e()
        attempts.append({"value_ms_per_step": round(ms_total / K, 5), "e2e_ms_per_step": round(e2e_ms / K, 5)})
        if abs(ms_total - e2e_ms) <= 0.15 * min(ms_total, e2e_ms):
            break
    agreement = abs(ms_total - e2e_ms) / min(ms_total, e2e_ms)
    ms_per_step = ms_total / K
    value = light_rays / (ms_total * 1e-3) / 1e6
    e2e_value = light_rays / (e2e_ms * 1e-3) / 1e6
    t_load_end = time.time()
    if rank == 0:
        sampler.stop()
    clocks = sampler.window(t_load_begin, t_load_end) if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dev.readback(L.OUT_TONE_MAPPED))     # frame W + K, the last of both timed arms

    # ------------------------------------------------ N > 1: is the frame the ranks assembled the frame one GPU renders?
    # Outside every timed region.  Frames 1..3 from zeroed state through the same tiles + frame assembly as the timed loop; rank 0
    # reads the assembled frame, renders the same three frames unsharded on its own GPU and compares byte for byte (and with the
    # hash committed in tests/golden/frame_hashes.json for this config and build, if there is one).
    frame_check = None
    if world_size > 1 and frame_targets and not args.no_frame_check:
        import hashlib
        dev.set_profiling(False, False)
        dev.reset_temporal_state()
        frame_no[0] = 0
        CHECK_FRAMES = 3
        for n in range(CHECK_FRAMES):
            begin_frame()
            dev.render_frame(inputs[n])
            gather_frame()
        barrier()
        if rank == 0:
            assembled = dev.frame_read(frame_targets[(frame_no[0] - 1) & 1])
            frame_check = {"frames": CHECK_FRAMES, "assembled_sha256": hashlib.sha256(assembled.tobytes()).hexdigest()}
            try:
                full = plugin.HikariPlugin(W, H, cuda_device=local_rank)
                full.upload_scene(world)
                for n in range(CHECK_FRAMES):
                    full.render_frame(inputs[n])
                unsharded = full.readback(L.OUT_TONE_MAPPED)
                full.close()
                frame_check["unsharded_sha256"] = hashlib.sha256(unsharded.tobytes()).hexdigest()
                frame_check["identical"] = bool(assembled.tobytes() == unsharded.tobytes())
                if not frame_check["identical"]:
                    frame_check["differing_pixels"] = int(np.any(assembled != unsharded, axis=-1).sum())
            except Exception as e:       # e.g. not enough memory for an unsharded 8K context next to the tile
                frame_check["unsharded_error"] = str(e)[:200]
            stored = stored_frame_hash(args.config, CHECK_FRAMES)
            if stored:
                frame_check["stored_sha256"] = stored
                frame_check["matches_stored"] = stored == frame_check["assembled_sha256"]
        barrier()
    elif world_size == 1 and args.print_frame_hash:
        import hashlib
        dev.set_profiling(False, False)
        dev.reset_temporal_state()
        for n in range(3):
            dev.render_frame(inputs[n])
        frame_check = {"frames": 3, "unsharded_sha256": hashlib.sha256(dev.readback(L.OUT_TONE_MAPPED).tobytes()).hexdigest()}

    # ------------------------------------------------ animated scene: cost of the per-frame scene half (not in `value`)
    # one instance moves -> previous_transform_system + prepare_instances on the host (TLAS, emissive BVH, alias tables;
    # instance.rs:352-437) and hk_scene_update_instances (H2D of the instance-level buffers)
    scene_update = None
    if world_size == 1:
        base = np.array(scene.inst_transform[len(scene.inst_transform) - 1], np.float32)
        host_ms, upload_ms = [], []
        for n in range(12):
            moved = base.copy()
            moved[12] += 0.001 * (n + 1)
            t0 = time.perf_counter()
            world.set_instance_transform(len(scene.inst_transform) - 1, moved)
            world.previous_transform_system()
            world.prepare_instances()
            t1 = time.perf_counter()
            dev.update_instances(world)
            t2 = time.perf_counter()
            host_ms.append((t1 - t0) * 1e3); upload_ms.append((t2 - t1) * 1e3)
        # the same motion through the device-side rebuild (hk_scene_update_transforms, csrc/kernels_scene.cu): host time of the call
        # (pinned staging + 4 launches, no synchronisation unless rays walk the 4-wide trees) and time until the kernels have run
        call_ms, done_ms, on_device = [], [], True
        for n in range(12):
            moved = base.copy()
            moved[12] += 0.001 * (n + 13)
            dev.sync()
            t0 = time.perf_counter()
            world.set_instance_transform(len(scene.inst_transform) - 1, moved)
            world.previous_transform_system()
            on_device = dev.update_transforms(world) and on_device
            t1 = time.perf_counter()
            dev.sync()
            t2 = time.perf_counter()
            call_ms.append((t1 - t0) * 1e3); done_ms.append((t2 - t0) * 1e3)
        world.prepare_instances()          # leave the host mirror's buffers describing the scene on the device
        dev.update_instances(world)
        d = world.scene_desc()
        scene_update = {"host_rebuild_ms": round(float(np.median(host_ms[2:])), 4), "upload_ms": round(float(np.median(upload_ms[2:])), 4),
                        "device_rebuild_call_ms": round(float(np.median(call_ms[2:])), 4),
                        "device_rebuild_done_ms": round(float(np.median(done_ms[2:])), 4), "device_path_taken": bool(on_device),
                        "instances": int(d.instance_count), "tlas_nodes": int(d.instance_node_count), "alias_entries": int(d.alias_count),
                        "note": "per-frame cost when instances move, host path (prepare_instances + hk_scene_update_instances) against "
                                "the device-side rebuild (hk_scene_update_transforms: call returns / kernels done); outside the timed "
                                "region of value / e2e (static benchmark scene)"}

    if rank != 0:
        if world_size > 1:
            dist.destroy_process_group()
        return

    # ---------------------------------------------------------------- roofline of the dominant kernel
    peak, peak_kind = peaks()
    signals = 3 if settings.indirect_bounces else 2
    ran = [(kernel_ms[i], name) for i, name in enumerate(L.KERNEL_NAMES) if kernel_ms[i] > 0]
    dom = L.KERNEL_NAMES[dominant]
    # N = 1: the dominant kernel's duration measured LIVE inside the timed region (mean over its K launches, 2 event records per
    # frame); N > 1: from the per-kernel replay of the same frames on this rank
    dom_ms = dom_live if dom_live else float(kernel_ms[dominant])
    rows_launched = {"gbuffer": 36, "direct": 36, "emissive": 36, "indirect": 36, "emissive_spatial": 16, "indirect_spatial": 16,
                     "demodulation": 15, "denoise_0": 7, "denoise_1": 3, "denoise_2": 1, "denoise_3": 0, "tone_mapping": 0}
    def launch_pixels(name):
        g = rows_launched[name]
        return (min(H, r1 + g) - max(0, r0 - g)) * (min(W, x1 + g) - max(0, x0 - g))
    bpp = BYTES_PER_PIXEL[dom] * (signals if dom in PER_SIGNAL else 1)
    if dom == "denoise_3":
        bpp += BYTES_PER_PIXEL["tone_mapping"]      # fused tone mapping
    alg_bytes = bpp * launch_pixels(dom)
    achieved = alg_bytes / (dom_ms * 1e-3) / 1e9
    frame_bpp = sum(BYTES_PER_PIXEL[name] * (signals if name in PER_SIGNAL else 1) for _, name in ran)
    if kernel_ms[L.KERNEL_NAMES.index("tone_mapping")] == 0:
        frame_bpp += BYTES_PER_PIXEL["tone_mapping"]
    frame_achieved = frame_bpp * W * H / (ms_per_step * 1e-3) / 1e9

    traffic = None   # measured DRAM bytes per launch of the dominant kernel, from the committed ncu capture of this workload
    try:
        if world_size == 1:
            with open(os.path.join(ROOT, "profiles", "r2_dram_traffic.json")) as f:
                traffic = json.load(f).get(args.config, {}).get(dom)
    except Exception:
        traffic = None
    out = {
        "metric": "Mrays/s", "value": round(value, 3), "unit": "Mrays/s", "n_gpus": world_size, "steps": K, "warmup": W_,
        "ms_per_step": round(ms_per_step, 5), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": f"reference assets ({ASSET_OF[cfg['scene']]}) + blue-noise seed (no synthetic inputs exist for this path)",
        "config": dict(config_json(args.config, cfg, settings, world_size, args.gather), tiles=[list(t) for t in tiles],
                       **({"halo_margin": args.halo_margin} if (world_size > 1 and args.halo_margin is not None) else {}),
                       **({"camera": "translating (0.003, 0.001, -0.002) per frame"} if args.moving_camera else {})),
        "rays_per_frame": {"light_tlas": rays[1] / K, "light_blas": rays[2] / K, "primary": rays[0] / K},
        "fps": round(1e3 / ms_per_step, 2),
        "e2e": {"value": round(e2e_value, 3), "unit": "Mrays/s", "ms_per_step": round(e2e_ms / K, 5),
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h_bytes},
        "gpu_launches": int(launches_per_frame * K),
        "kernel_ms": {name: round(float(kernel_ms[i]), 5) for i, name in enumerate(L.KERNEL_NAMES) if kernel_ms[i] > 0},
        "kernel_ms_source": "replay of the timed frames with every kernel bracketed by CUDA events (outside the timed region)",
        "frame_ms": {"min": round(min(per_frame), 5), "median": round(float(np.median(per_frame)), 5), "max": round(max(per_frame), 5),
                     "note": "per-frame CUDA-event times of the timed region on rank 0"},
        "value_vs_e2e": {"relative_difference": round(agreement, 4), "within_15_percent": bool(agreement <= 0.15), "attempts": attempts},
        "roofline": {"bound": "hbm", "kernel": dom, "kernel_ms": round(dom_ms, 5),
                     "kernel_ms_source": "live, timed region" if dom_live else "replay",
                     "achieved": round(achieved, 2), "peak": peak, "unit": "GB/s",
                     "frac": round(achieved / peak, 5), "traffic": traffic, "peak_source": f"MEASURED_PEAKS.json ({peak_kind})",
                     "algorithmic_bytes_per_launch": int(alg_bytes),
                     "frame": {"bytes_per_pixel": frame_bpp, "achieved": round(frame_achieved, 2),
                               "frac": round(frame_achieved / peak, 5)}},
        "clocks": clocks,
    }
    if scene_update:
        out["scene_update"] = scene_update
    if frame_check:
        out["frame_check"] = frame_check
    if world_size == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline_sample(args.config, seconds_budget=25.0)
    print(json.dumps(out), flush=True)
    if world_size > 1:
        dist.destroy_process_group()


DUMP_LIMIT = 64_000_000    # bytes --dump-outputs may write, .npy header included
NPY_HEADER = 4096          # room kept for the header np.save writes (128 bytes for these arrays)


def dump_outputs(directory, tone_mapped):
    """--dump-outputs: the tone-mapped image of the last timed step (what render_frame / run_frame hand a caller), as float32
    DIR/tone_mapped.npy (H x W x 4).  An image that does not fit DUMP_LIMIT is replaced by a fixed sample of its pixels (seed 0, sorted
    pixel order): DIR/tone_mapped_sample.npy (n x 4)."""
    img = np.asarray(tone_mapped, np.float32)
    name = "tone_mapped"
    budget = DUMP_LIMIT - NPY_HEADER
    if img.nbytes > budget:
        px = img.reshape(-1, img.shape[-1])
        keep = np.sort(np.random.default_rng(0).choice(px.shape[0], budget // px[0].nbytes, replace=False))
        img, name = px[keep], "tone_mapped_sample"
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, name + ".npy"), img)


# ============================================================================================ CPU arms
def stored_frame_hash(config, frames):
    """sha256 of the tone-mapped frame `frames` of `config` rendered unsharded on one GPU with the default build, committed by
    tools/record_frame_hashes (tests/golden/frame_hashes.json); None when there is none"""
    try:
        with open(os.path.join(ROOT, "tests", "golden", "frame_hashes.json")) as f:
            return json.load(f).get(f"{config}:frame{frames}")
    except Exception:
        return None


def host_threads():
    """usable host cores: affinity mask, capped by the cgroup CPU quota (os.cpu_count() reports the whole machine)"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period))))
    except Exception:
        try:
            quota = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota > 0:
                n = min(n, max(1, quota // period))
        except Exception:
            pass
    return max(1, n)


_BEST_THREADS = {}


def best_threads(config, width, height):
    """The host may expose more hardware threads than the container can actually use; time one oracle frame at
    n, n/2, n/4 ... threads and keep the fastest, so the CPU arm is reported at its best."""
    key = (config, width, height)
    if key in _BEST_THREADS:
        return _BEST_THREADS[key]
    from bevy_hikari_b200 import plugin
    n = host_threads()
    cands = []
    while n >= 1:
        cands.append(n)
        if n <= 4:
            break
        n //= 2
    best, best_t = cands[-1], float("inf")
    for t in cands:
        orc, settings, view, pview, lights = oracle_for(config, width, height, threads=t, calibrate=False)
        inp = plugin.make_frame_inputs(settings, 1, view, pview, lights)
        orc.render_frame(inp)
        t0 = time.perf_counter()
        orc.render_frame(plugin.make_frame_inputs(settings, 2, view, pview, lights))
        dt = time.perf_counter() - t0
        orc.close()
        if dt < best_t:
            best, best_t = t, dt
    _BEST_THREADS[key] = best
    return best


def oracle_for(config, width, height, threads=None, calibrate=True):
    if threads is None:
        threads = best_threads(config, width, height) if calibrate else host_threads()
    from bevy_hikari_b200 import plugin, scenes
    from oracle import oracle
    cfg = scenes.CONFIGS[config]
    scene = scenes.SCENE_BUILDERS[cfg["scene"]]()
    world = scene.populate(plugin.World())       # host-side scene preparation only; no CUDA call
    view, pview, lights = scene.view_inputs(width, height)
    settings = scenes.config_settings(config)
    orc = oracle.Oracle(width, height, plugin.load_noise(), threads)
    orc.upload_scene_desc(world.scene_desc())
    return orc, settings, view, pview, lights


def cpu_baseline_sample(config, seconds_budget):
    """The oracle on the host cores, on a bounded sample: frames 1.. of the same scene / settings at 1/4 x 1/4 of the
    resolution (rays per pixel do not depend on resolution), as many frames as fit in the budget (at least 2)."""
    from bevy_hikari_b200 import plugin, scenes
    cfg = scenes.CONFIGS[config]
    w, h = cfg["width"] // 4, cfg["height"] // 4
    orc, settings, view, pview, lights = oracle_for(config, w, h)
    rays, frames, t_total = 0.0, 0, 0.0
    n = 1
    while frames < 2 or (t_total < seconds_budget and frames < 64):
        inp = plugin.make_frame_inputs(settings, n, view, pview, lights)
        t0 = time.perf_counter()
        orc.render_frame(inp)
        dt = time.perf_counter() - t0
        st = orc.stats()
        if n > 1:   # frame 1 is warm-up (page faults)
            rays += st.tlas_rays + st.blas_rays
            t_total += dt
            frames += 1
        n += 1
    return {"value": round(rays / t_total / 1e6, 4), "unit": "Mrays/s", "cores": orc.threads, "kind": "port",
            "ms_per_frame_sample": round(t_total / frames * 1e3, 2),
            "sample": f"{frames} frames of {config} at {w}x{h} (1/16 of the pixels, same scene/settings/frame sequence), "
                      f"oracle = C++/OpenMP restatement of the reference WGSL, bit-identical to the reference's shader text executed on the CPU (tests/golden/wgsl_*.npz); the reference itself (Rust+wgpu) cannot be built offline"}


def reference_sample_size(config, W_, K, budget_s=150.0):
    """The reference arm renders the TRUE configuration when W + K frames of it fit the time budget on this box's host cores;
    otherwise the largest of 1/2, 1/4, 1/8 of the resolution (per axis) that does.  Estimated from one frame at 1/8 resolution
    (cost per pixel is resolution independent for this path)."""
    from bevy_hikari_b200 import plugin, scenes
    cfg = scenes.CONFIGS[config]
    W, H = cfg["width"], cfg["height"]
    pw, ph = max(W // 8, 16), max(H // 8, 16)
    orc, settings, view, pview, lights = oracle_for(config, pw, ph)
    orc.render_frame(plugin.make_frame_inputs(settings, 1, view, pview, lights))
    t0 = time.perf_counter()
    orc.render_frame(plugin.make_frame_inputs(settings, 2, view, pview, lights))
    per_pixel = (time.perf_counter() - t0) / (pw * ph)
    orc.close()
    for div in (1, 2, 4, 8):
        w, h = W // div, H // div
        if per_pixel * w * h * (W_ + K) <= budget_s or div == 8:
            return w, h, div


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from bevy_hikari_b200 import plugin, scenes       # host mirror only (libhikari_host.so): no CUDA library is mapped by this arm
    cfg = scenes.CONFIGS[args.config]
    W_, K = args.warmup, args.steps
    w, h, div = reference_sample_size(args.config, W_, K)
    orc, settings, view, pview, lights = oracle_for(args.config, w, h)
    for n in range(1, W_ + 1):
        orc.render_frame(plugin.make_frame_inputs(settings, n, view, pview, lights))
    orc.stats()
    rays = 0.0
    t0 = time.perf_counter()
    for n in range(W_ + 1, W_ + K + 1):
        orc.render_frame(plugin.make_frame_inputs(settings, n, view, pview, lights))
        st = orc.stats()
        rays += st.tlas_rays + st.blas_rays
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        from bevy_hikari_b200 import layout as L
        dump_outputs(args.dump_outputs, orc.readback(L.OUT_TONE_MAPPED))
    value = rays / dt / 1e6
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    full = div == 1
    sample = ((f"each step = one frame of {args.config} at its full {w}x{h}" if full else
               f"each step = one frame of {args.config} rendered at {w}x{h} (1/{div * div} of the configuration's {cfg['width']}x{cfg['height']} "
               f"pixels, the largest size whose {W_ + K} frames fit the time budget on these cores; rays per pixel do not depend on resolution)") +
              "; CPU restatement of the reference WGSL (oracle/hk_oracle.cpp, OpenMP) — the reference's own wgpu path needs rustc + a Vulkan "
              "ICD, neither exists offline")
    config = config_json(args.config, cfg, settings, world_size)
    config["rendered_width"], config["rendered_height"], config["rendered_pixel_fraction"] = w, h, round(1.0 / (div * div), 6)
    ms_step = dt / K * 1e3
    out = {"impl": "reference", "metric": "Mrays/s", "value": round(value, 4), "unit": "Mrays/s", "n_gpus": args.gpus, "steps": K,
           "warmup": W_, "ms_per_step": round(ms_step, 3),
           "ms_per_step_note": ("full configuration" if full else f"for the {w}x{h} sample; x{div * div} for the configuration's pixel count"),
           "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "f32", "data": f"reference assets ({ASSET_OF[cfg['scene']]}) + blue-noise seed",
           "config": config,
           "cpu_baseline": {"value": round(value, 4), "unit": "Mrays/s", "cores": orc.threads, "kind": "port", "sample": sample},
           "e2e": {"value": round(value, 4), "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "libraries": "oracle/libhk_oracle.so + bevy_hikari_b200/libhikari_host.so (scene preparation); the CUDA library is not loaded",
           "mapped_cuda_library": any("libhikari_b200" in l for l in open("/proc/self/maps"))}
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--config", default="cornell_1080p")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--equal-tiles", action="store_true", help="N > 1: equal grid of tiles instead of cost-balanced strips")
    ap.add_argument("--moving-camera", action="store_true", help="translate the camera every frame (temporal reprojection crosses tile borders)")
    ap.add_argument("--halo-margin", type=int, default=None,
                    help="N > 1: exact tiling under camera motion — ghost ring of 36 + M pixels and a halo pull after every frame")
    ap.add_argument("--no-frame-check", action="store_true", help="N > 1: skip the assembled-frame == unsharded-frame check")
    ap.add_argument("--print-frame-hash", action="store_true", help="N = 1: add the sha256 of frame 3 (for tests/golden/frame_hashes.json)")
    ap.add_argument("--lib", default=None, help="tuning: load this build of libhikari_b200.so (tools/build_variants.py) instead of the in-tree one")
    ap.add_argument("--gather", default="peer", choices=["peer", "nccl"],
                    help="N > 1: peer = tiles stored straight into rank 0's frame over NVLink (CUDA IPC); nccl = all_gather of tiles")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the tone-mapped image of the last timed step to DIR as float32 .npy (at most 64 MB: a fixed sample of "
                         "the pixels of larger images); --gpus 1 only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.gpus > 1:
        ap.error("--dump-outputs: --gpus 1 only")
    args.warmup = max(args.warmup, 3)
    if args.lib:
        from bevy_hikari_b200 import _ffi
        _ffi.LIB_PATH = os.path.abspath(args.lib)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
