#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native compositor (contract: see DESIGN.md section 6).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg3] [--impl ours|reference]

A "step" is one pass of the hot path over one batch of synthetic input: one output frame of the
workload (default: BASELINE config 3, 16 x 4K NV12 -> 4K NV12 mosaic with per-input Lanczos3 4:1
downscale, rounded corners and an alpha overlay).  N > 1: one process per GPU (torchrun), every rank
composites its own output stream (weak scaling, no data-path collective: outputs shard, SURVEY 8e).

`value`     frames/s with inputs resident in HBM, device-timed (CUDA events on the launching stream).
`e2e`       frames/s through the C ABI with pinned HOST buffers (H2D + kernels + D2H inside the timing).
`roofline`  dominant kernel: algorithmic bytes per launch / its device time (events inside the library).
`cpu_baseline` / `--impl reference`: the CPU oracle (restatement of the reference's wgpu path; the
            reference itself is Rust + wgpu and cannot run here) timed on the host cores, bounded sample.

--dump-outputs DIR  after the timed steps, writes the output planes of the last timed step as DIR/<name>.npy
            (float32 copies of the NV12 bytes, e.g. output_1_y.npy (H, W) and output_1_uv.npy (H/2, W/2, 2)).  Inputs
            are seeded, so the same arguments give the same inputs on every run and two builds can be compared file by
            file.  At most 64 MB are written: a larger output keeps a fixed, seeded subset of its rows (the row numbers
            go to <name>_rows.npy).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np

BG = (0x33, 0x33, 0x33, 255)


# ------------------------------------------------------------------------------------------------
# workloads (BASELINE.json configs / SURVEY 8d)
# ------------------------------------------------------------------------------------------------
def workload(name):
    import smelter_b200 as s
    V = s.ViewComponent
    bg = s.RGBAColor(*BG)

    def streams(n):
        return [s.InputStreamComponent(input_id=f"input_{i}") for i in range(1, n + 1)]

    def rounded_tiles(n, radius, shadow=False):
        kids = []
        for c in streams(n):
            sh = [s.BoxShadow(6.0, 6.0, 16.0, s.RGBAColor(0, 0, 0, 160))] if shadow else []
            kids.append(s.RescalerComponent(child=c, border_radius=s.BorderRadius.new_with_radius(radius), box_shadow=sh))
        return kids

    if name == "cfg3":   # 16 x 4K NV12 -> 4K NV12, Tiles 4x4 (scale exactly 4 -> 25-tap Lanczos3), GpuOptimized
        W, H, n, iw, ih = 3840, 2160, 16, 3840, 2160
        overlay = V(position=s.Position.Absolute(width=1600.0, height=360.0, left=1120.0, bottom=120.0),
                    background_color=s.RGBAColor(16, 32, 160, 112), border_radius=s.BorderRadius.new_with_radius(48.0))
        scene = V(background_color=bg, children=[s.TilesComponent(children=rounded_tiles(n, 32.0), background_color=bg),
                                                 overlay])
        mode = s.RenderingMode.GpuOptimized
        desc = "16x(3840x2160 NV12)->3840x2160 NV12, Tiles 4x4, Lanczos3 4:1, rounded corners + alpha overlay, GpuOptimized"
    elif name == "cfg3b":  # same with 1080p inputs (scale 2)
        W, H, n, iw, ih = 3840, 2160, 16, 1920, 1080
        overlay = V(position=s.Position.Absolute(width=1600.0, height=360.0, left=1120.0, bottom=120.0),
                    background_color=s.RGBAColor(16, 32, 160, 112), border_radius=s.BorderRadius.new_with_radius(48.0))
        scene = V(background_color=bg, children=[s.TilesComponent(children=rounded_tiles(n, 32.0), background_color=bg),
                                                 overlay])
        mode = s.RenderingMode.GpuOptimized
        desc = "16x(1920x1080 NV12)->3840x2160 NV12, Tiles 4x4, Lanczos3 2:1, rounded corners + alpha overlay"
    elif name == "grid25":  # 25 x 4K -> 4K, Tiles 5x5: ratio 5:1 > 4 -> one box pre-decimation level + Lanczos (the generic path)
        W, H, n, iw, ih = 3840, 2160, 25, 3840, 2160
        scene = s.TilesComponent(children=streams(n), background_color=bg)
        mode = s.RenderingMode.GpuOptimized
        desc = "25x(3840x2160 NV12)->3840x2160 NV12, Tiles 5x5, box 2:1 + Lanczos3 2.5:1 (resampler.rs:56-67), GpuOptimized"
    elif name == "cfg2":  # 4 x 1080p NV12 -> 1080p NV12, Tiles 2x2, CpuOptimized (gamma blend, bilinear)
        W, H, n, iw, ih = 1920, 1080, 4, 1920, 1080
        scene = s.TilesComponent(children=streams(n), background_color=bg)
        mode = s.RenderingMode.CpuOptimized
        desc = "4x(1920x1080 NV12)->1920x1080 NV12, Tiles 2x2, bilinear, CpuOptimized"
    elif name == "cfg5":  # 32 x 4K -> 8K, box shadow + radius
        W, H, n, iw, ih = 7680, 4320, 32, 3840, 2160
        scene = s.TilesComponent(children=rounded_tiles(n, 40.0, shadow=True), background_color=bg, margin=24.0)
        mode = s.RenderingMode.GpuOptimized
        desc = "32x(3840x2160 NV12)->7680x4320 NV12, Tiles 6x6 grid, Lanczos3 + box-shadow + radius"
    elif name == "cfg4":  # 64 outputs x 1080p (4 of 8 pooled inputs each), 8 per GPU, shared inputs broadcast over NVLink
        W, H, n, iw, ih = 1920, 1080, 8, 1920, 1080
        scene = None   # per-rank scenes are built in main(): output k uses inputs (k + j) % 8, j < 4
        mode = s.RenderingMode.GpuOptimized
        desc = ("8 outputs/GPU of 4x(1920x1080 NV12)->1920x1080 NV12 Tiles 2x2 Lanczos3 2:1, inputs from a pool of 8 "
                "shared by every GPU over NVLink each tick (config.secondary.exchange: ncclBroadcast / copy-engine pull / read in place)")
    elif name == "passthrough":  # single_video_pass_through of the reference's benchmark suite
        W, H, n, iw, ih = 3840, 2160, 1, 3840, 2160
        scene = s.InputStreamComponent(input_id="input_1")
        mode = s.RenderingMode.GpuOptimized
        desc = "1x(3840x2160 NV12)->3840x2160 NV12 pass-through root"
    else:
        raise SystemExit(f"unknown workload {name}")
    n_out = 8 if name == "cfg4" else 1
    # SURVEY 8d: every needed input byte once (shared inputs count once per GPU per tick) + every output byte once
    alg = n * (iw * ih * 3 // 2) + n_out * (W * H * 3 // 2)
    tiles = 4 if name == "cfg4" else n   # texture layers per output frame (the CPU baseline times one of them)
    return dict(name=name, scene=scene, W=W, H=H, n=n, iw=iw, ih=ih, mode=mode, desc=desc, alg_bytes=alg, n_out=n_out,
                tiles=tiles)


def cfg4_scene(g, n=8):
    """scene of global output g of BASELINE config 4: Tiles 2x2 of inputs (g + j) % n, j < 4, from the pool of n"""
    import smelter_b200 as s
    kids = [s.InputStreamComponent(input_id=f"input_{(g + j) % n + 1}") for j in range(4)]
    return s.TilesComponent(children=kids, background_color=s.RGBAColor(*BG))


# ------------------------------------------------------------------------------------------------
def synth_planes_torch(torch, dev, w, h, seed):
    """procedural NV12 frame on the device: smooth blobs + noise, legal range."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    def plane(pw, ph, lo, hi, ch):
        coarse = torch.rand((ph // 32 + 2, pw // 32 + 2, ch), generator=g, device=dev)
        up = coarse.repeat_interleave(32, 0).repeat_interleave(32, 1)[:ph, :pw]
        x = up * 0.85 + 0.15 * torch.rand((ph, pw, ch), generator=g, device=dev)
        return (lo + x * (hi - lo)).to(torch.uint8).contiguous()
    return plane(w, h, 16, 235, 1), plane(w // 2, h // 2, 16, 240, 2)


SETUP_SECONDS = 0.3   # untimed set-up ticks before the W warm-up steps (clock ramp, tables, descriptors)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,clocks.mem,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, indices):
        indices = list(indices)
        self.index, self.rows, self.proc, self.n = ",".join(str(i) for i in indices), [], None, len(indices)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "20" if self.n == 1 else "50"],   # a query of 8 GPUs
                                         stdout=subprocess.PIPE, text=True)                               # holds driver locks for longer
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def mark(self):
        """the timed region starts here: only rows that arrive from now on are reported"""
        self.i0 = len(self.rows)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        i1 = len(self.rows)
        i0 = min(getattr(self, "i0", 0), max(i1 - self.n, 0))   # a region shorter than one sampling period: the latest row per GPU
        self.rows = self.rows[i0:i1] if i1 > i0 else self.rows[-self.n:]
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        ok = [r for r in self.rows if len(r) > 8 and r[1].replace(".", "").isdigit()]
        per_gpu = {}
        for r in ok:
            per_gpu.setdefault(r[0], []).append(float(r[1]))
        med = {g: float(np.median(v)) for g, v in per_gpu.items()}
        mx = [float(r[2]) for r in ok if r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in ok for n, v in zip(names, r[5:9]) if v == "Active"})
        # every GPU of the job is sampled; the reported clock is the slowest GPU's median under load
        return {"sm_mhz": min(med.values()) if med else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": min((len(v) for v in per_gpu.values()), default=0),
                "per_gpu_sm_mhz": [med[g] for g in sorted(med, key=int)] if len(med) > 1 else None}


# ------------------------------------------------------------------------------------------------
# CPU baseline: the oracle on a bounded sample (1 of n tiles of the workload)
# ------------------------------------------------------------------------------------------------
def metric_name(wl):
    """one string for both arms (the driver divides the two lines only when the metric strings agree)"""
    return "4K composited frames/sec (16-input grid) per GPU" if wl["name"] == "cfg3" else "composited output frames/sec"


def cpu_team():
    """fixed rule, identical in both arms: one OpenMP thread per physical core (half the logical CPUs of the affinity
    mask on an SMT box; every CPU when there are few)"""
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    return max(1, ncpu // 2) if ncpu >= 8 else max(1, ncpu)


CPU_TILES = 4   # distinct tiles per bounded sample


def cpu_steps(wl, steps, warmup):
    """Time the oracle on a BOUNDED SAMPLE of the workload: CPU_TILES distinct inputs, each composited into ITS
    tile-sized output region with the tile's layers (K1/K2 -> Lanczos -> K9 -> K11).  One step = one pass over the
    sample; its frame-time estimate = (sum of the tile times) x n_tiles / CPU_TILES.  Returns (list of per-step frame
    times in seconds, description, threads)."""
    import smelter_b200 as s
    from oracle import oracle as orc
    from tests import harness
    n, iw, ih = wl["tiles"], wl["iw"], wl["ih"]
    cols = int(np.ceil(np.sqrt(n)))
    tw, th = wl["W"] // cols, (wl["W"] // cols) * 9 // 16
    if wl["name"] == "passthrough":
        tw, th = wl["W"], wl["H"]
    k = min(CPU_TILES, n)
    tiles_in = []
    for t in range(k):
        y, u, v = harness.smooth_yuv420(1 + t, iw, ih)
        tiles_in.append((y, np.stack([u, v], axis=-1)))
    mode = orc.MODE_CPU_OPTIMIZED if wl["mode"] == s.RenderingMode.CpuOptimized else orc.MODE_GPU_OPTIMIZED
    radius = 0.0 if wl["name"] in ("cfg2", "passthrough") else 32.0
    layers = [orc.make_layout(orc.LAYOUT_COLOR, 0, 0, tw, th, color=BG),
              orc.make_layout(orc.LAYOUT_TEXTURE, 0, 0, tw, th, child_index=0, crop=(0, 0, iw, ih),
                              masks=[((radius,) * 4, 0, 0, tw, th)] if radius else [])]
    if wl["name"] in ("cfg3", "cfg3b"):  # this tile's share of the alpha overlay
        layers.append(orc.make_layout(orc.LAYOUT_COLOR, th * 0.3, 0, tw, th * 0.5, color=(16, 32, 160, 112)))

    def once(y, uv):
        t0 = time.perf_counter()
        node = orc.nv12_to_rgba(y, uv, iw, ih)
        img = node if wl["name"] == "passthrough" else orc.render_layout_node(tw, th, layers, [node], mode=mode)
        orc.rgba_to_nv12(img)
        return time.perf_counter() - t0

    orc.set_num_threads(cpu_team())
    out = []
    for i in range(warmup + steps):
        dt = sum(once(y, uv) for (y, uv) in tiles_in) * n / k
        if i >= warmup:
            out.append(dt)
    desc = (f"{k} of {n} tiles per step: each one {iw}x{ih} NV12 input -> {tw}x{th} NV12 region with the tile's layers; "
            f"frame time = {n}/{k} x the step's tile times; value = 1 / median over the steps; "
            f"OpenMP team = 1 thread per physical core")
    return out, desc, orc.num_threads()


def run_reference(args, wl):
    """--impl reference: the reference's own CPU path cannot run here (Rust + wgpu, no rustc / Vulkan ICD in
    the image), so this arm times the CPU oracle -- the restatement of that path -- on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    times, desc, cores = cpu_steps(wl, args.steps, args.warmup)
    per_frame = float(np.median(times))
    fps = 1.0 / per_frame
    line = {"impl": "reference", "metric": metric_name(wl), "value": fps, "unit": "frames/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_frame * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 math on u8 planes (f16 resampler scratch)",
            "data": "synthetic",
            "config": {"workload": wl["name"], "detail": wl["desc"]},
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port", "sample": desc,
                             "spread": {"min_ms": float(np.min(times)) * 1e3, "max_ms": float(np.max(times)) * 1e3, "steps": len(times)}},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


DUMP_BYTES = 64 * 10**6   # the whole --dump-outputs set, .npy headers included


def dump_outputs(directory, planes, budget=DUMP_BYTES):
    """planes: {name: uint8 numpy array (rows first)}.  Writes each as float32 <name>.npy; when the set would exceed the
    budget, every plane keeps the same seeded share of its rows and the chosen row numbers are written beside it."""
    os.makedirs(directory, exist_ok=True)
    header = 256   # per file, generous for an .npy header
    total = sum(p.size * 4 + header for p in planes.values())
    share = 1.0 if total <= budget else (budget - 2 * header * len(planes)) / (total + 8 * sum(len(p) for p in planes.values()))
    for i, (name, p) in enumerate(planes.items()):
        if share < 1.0:
            rows = np.sort(np.random.default_rng(1000 + i).choice(len(p), max(1, int(len(p) * share)), replace=False))
            np.save(os.path.join(directory, f"{name}_rows.npy"), rows.astype(np.float64))
            p = p[rows]
        np.save(os.path.join(directory, f"{name}.npy"), p.astype(np.float32))


class _DevMem:
    """a raw device range as a CUDA array (torch.as_tensor views it without copying)"""
    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


def measure_cfg4(torch, dist, dev, rank, world, local, steps, warmup, exchange="nccl"):
    """BASELINE config 4 on the running process group: 8 outputs per GPU; every tick the pool of 8 shared 1080p inputs,
    ingested round-robin by the GPUs, has to reach every GPU.  exchange:
      nccl         smr_comm_exchange_inputs: ncclBroadcast of the pooled planes on the communication stream
      peer_copy    smr_comm_pull_inputs: copy-engine pulls out of the roots' IPC-mapped pools after a 4-byte all-reduce
      peer_direct  nothing is copied: the fused resample kernel's TMA loads read the roots' pools over NVLink
    Returns the device-timed aggregate frames/s (max over ranks) and the bytes that cross NVLink per tick."""
    import smelter_b200 as s
    from smelter_b200 import _ffi as F
    wl = workload("cfg4")
    n, iw, ih, W, H, n_out = wl["n"], wl["iw"], wl["ih"], wl["W"], wl["H"], wl["n_out"]
    peer = exchange in ("peer_copy", "peer_direct") and world > 1
    nvar = 3 if exchange == "peer_direct" else 2   # header: a directly read pool set may be rewritten three ticks later
    r = s.Renderer(s.RendererOptions(rendering_mode=wl["mode"], cuda_device=local))
    ids = [f"input_{i}".encode() for i in range(1, n + 1)]
    for b in ids:
        r.register_input(b.decode())
    out_ids = [f"output_{k + 1}".encode() for k in range(n_out)]
    for k in range(n_out):
        r.update_scene(out_ids[k].decode(), s.Resolution(W, H), s.OutputFrameFormat.Nv12WgpuTexture, cfg4_scene(rank * n_out + k, n))
    roots = [i % world for i in range(n)]
    if world > 1:
        uid = [r.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        r.comm_init(uid[0], rank, world)
    order = sorted(range(n), key=lambda i: (roots[i], i))
    frames, arrs, peer_arrs, own_pools, opened = [], [], [], [], []
    for v in range(nvar):
        planes = [synth_planes_torch(torch, dev, iw, ih, 0x5EED4000 + 1000 * v + i + 97 * rank) for i in range(n)]
        nbytes = sum(t.numel() for i in order for t in planes[i])
        if peer:   # one pool per GPU, mappable by the other GPUs' handles; identical layout everywhere
            base, handle = r.peer_pool_alloc(nbytes)
            own_pools.append(base)
            pool = torch.as_tensor(_DevMem(base, nbytes), device=dev)
            handles = [None] * world
            dist.all_gather_object(handles, handle)
            bases = [base if k == rank else r.peer_pool_open(handles[k]) for k in range(world)]
            opened += [b for k, b in enumerate(bases) if k != rank]
        else:
            pool = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            base, bases = pool.data_ptr(), None
        off, packed, offs = 0, {}, {}
        for i in order:   # one pool per ingest GPU, identical layout on every rank (SMR_COMM_POOLED)
            views = []
            offs[i] = []
            for t in planes[i]:
                view = pool[off:off + t.numel()].view(t.shape)
                view.copy_(t)
                views.append(view)
                offs[i].append(off)
                off += t.numel()
            packed[i] = tuple(views)
        frames.append((pool, packed))

        def frame_array(base_of):
            arr = (F.InputFrame * n)()
            for k, i in enumerate(order):
                arr[k].input_id = ids[i]
                arr[k].format = F.FRAME_NV12
                arr[k].width, arr[k].height = iw, ih
                arr[k].mem_kind = F.MEM_DEVICE
                arr[k].planes[0], arr[k].planes[1] = base_of(i) + offs[i][0], base_of(i) + offs[i][1]
            return arr
        if exchange == "peer_direct" and world > 1:
            arrs.append(frame_array(lambda i: bases[roots[i]]))     # read in place: the root's pool
            peer_arrs.append(None)
        else:
            arrs.append(frame_array(lambda i: base))
            peer_arrs.append(frame_array(lambda i: bases[roots[i]]) if peer else None)
    comm_roots = [roots[i] for i in order]
    out_y = [torch.empty((H, W), dtype=torch.uint8, device=dev) for _ in range(n_out)]
    out_uv = [torch.empty((H // 2, W // 2, 2), dtype=torch.uint8, device=dev) for _ in range(n_out)]
    dev_out = (F.OutputFrame * n_out)()
    for k in range(n_out):
        dev_out[k].output_id = out_ids[k]
        dev_out[k].mem_kind = F.MEM_DEVICE
        dev_out[k].planes[0], dev_out[k].planes[1] = out_y[k].data_ptr(), out_uv[k].data_ptr()
    stream = torch.cuda.ExternalStream(r.cuda_stream(), device=dev)
    frame_ns = 33_333_333
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()

    def step(k):
        a = arrs[k % nvar]
        for f in a:
            f.pts_ns = k * frame_ns
        if world > 1:
            if exchange == "peer_copy":
                r.comm_pull_inputs(a, peer_arrs[k % nvar], n, comm_roots)
            else:
                r.comm_exchange_inputs(a, n, comm_roots, None, pooled=True, peer_direct=exchange == "peer_direct")
        r.render_raw(k * frame_ns, a, n, dev_out, n_out, wait=False)

    setup = 200   # a fixed count (the exchange is collective): tables, descriptors, arenas, load clocks -- then the W warm-up steps
    for k in range(setup + warmup):
        step(k)
        if k % 16 == 15:
            r.wait()
    r.wait()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for k in range(steps):
        step(setup + warmup + k)
    r.wait()
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    step(nvar * 100000)   # one more tick on frame set 0: its outputs must not depend on how the inputs travelled
    r.wait()
    torch.cuda.synchronize()
    digest = int(sum(int(t.to(torch.int64).sum().item()) * (j + 1) for j, t in enumerate(out_y + out_uv)))
    if dist is not None:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        dist.barrier()    # nobody unmaps a pool another rank may still be reading
    if world > 1:
        for b in opened:
            r.peer_pool_close(b)
        if dist is not None:
            dist.barrier()
        for b in own_pools:
            r.peer_pool_free(b)
        r.comm_destroy()
    moved = sum(iw * ih * 3 // 2 for i in range(n) if True) * (world - 1) if world > 1 else 0   # every input reaches the other N-1 GPUs
    return {"workload": "cfg4", "detail": wl["desc"], "exchange": exchange if world > 1 else "none",
            "value": world * n_out * steps / (ms * 1e-3), "unit": "frames/s",
            "ms_per_tick": ms / steps, "steps": steps, "outputs_per_gpu": n_out,
            "nvlink_broadcast_bytes_per_tick": moved, "scaling": "weak", "output_digest_rank": digest}


def measure_cfg4_modes(torch, dist, dev, rank, world, local, steps, warmup, modes):
    """the cfg4 leg under every requested exchange; the line carries the fastest, the others ride along"""
    res = {m: measure_cfg4(torch, dist, dev, rank, world, local, steps, warmup, exchange=m) for m in modes}
    digests = {m: res[m].pop("output_digest_rank") for m in modes}
    best = max(modes, key=lambda m: res[m]["value"])
    out = dict(res[best])
    out["modes"] = {m: {"value": res[m]["value"], "ms_per_tick": res[m]["ms_per_tick"]} for m in modes}
    same = torch.tensor([1 if len(set(digests.values())) == 1 else 0], device=dev)
    if dist is not None:
        dist.all_reduce(same, op=dist.ReduceOp.MIN)   # on every rank
    out["same_frames_in_every_mode"] = bool(same.item())
    return out


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3")
    ap.add_argument("--variants", type=int, default=4, help="distinct synthetic frames per input, cycled")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="N > 1: skip the cfg4 (NVLink exchange) leg")
    ap.add_argument("--exchange", default="all", choices=["all", "nccl", "peer_copy", "peer_direct"],
                    help="N > 1, cfg4 leg: how the shared inputs reach the other GPUs (all: measure each, report the fastest)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the output planes of the last timed step to DIR/<name>.npy (float32, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3)
    wl = workload(args.workload)
    if args.impl == "reference":
        run_reference(args, wl)
        return

    import torch
    import smelter_b200 as s
    from smelter_b200 import _ffi as F

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the compositor has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # nvidia-smi needs a few hundred ms before its first row: started now, it is streaming by the time the timed region
    # begins (rank 0 only -- its line is the one that is printed)
    clocks = ClockSampler(range(world) if world > 1 else [local])
    if int(os.environ.get("RANK", "0")) == 0:
        clocks.start()
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    r = s.Renderer(s.RendererOptions(rendering_mode=wl["mode"], cuda_device=local))
    n, iw, ih, W, H = wl["n"], wl["iw"], wl["ih"], wl["W"], wl["H"]
    ids = [f"input_{i}".encode() for i in range(1, n + 1)]
    for b in ids:
        r.register_input(b.decode())
    n_out = wl["n_out"]
    out_ids = [f"output_{k + 1}".encode() for k in range(n_out)]
    if wl["name"] == "cfg4":
        for k in range(n_out):
            r.update_scene(out_ids[k].decode(), s.Resolution(W, H), s.OutputFrameFormat.Nv12WgpuTexture,
                           cfg4_scene(rank * n_out + k, n))
    else:
        r.update_scene("output_1", s.Resolution(W, H), s.OutputFrameFormat.Nv12WgpuTexture, wl["scene"])
    # shared-input replication (only cfg4 has inputs referenced from several GPUs)
    roots = None
    if wl["name"] == "cfg4" and world > 1:
        uid = [r.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        r.comm_init(uid[0], rank, world)
        roots = [i % world for i in range(n)]   # input i is ingested on GPU i % N

    # ---- device-resident synthetic inputs: `variants` distinct frames per input, cycled -------------
    nvar = max(1, args.variants)
    dev_frames = [[synth_planes_torch(torch, dev, iw, ih, 0x5EED0000 + 1000 * v + i + 97 * rank) for i in range(n)]
                  for v in range(nvar)]
    out_y = [torch.empty((H, W), dtype=torch.uint8, device=dev) for _ in range(n_out)]
    out_uv = [torch.empty((H // 2, W // 2, 2), dtype=torch.uint8, device=dev) for _ in range(n_out)]

    def in_array(planes_for_variant, mem_kind, ptr):
        arr = (F.InputFrame * n)()
        for i in range(n):
            yv, uvv = planes_for_variant[i]
            arr[i].input_id = ids[i]
            arr[i].format = F.FRAME_NV12
            arr[i].width, arr[i].height = iw, ih
            arr[i].mem_kind = mem_kind
            arr[i].planes[0], arr[i].planes[1] = ptr(yv), ptr(uvv)
        return arr

    if roots is not None:
        # each ingest GPU keeps the frames it owns in one pool: the planes of a root are contiguous, so the library
        # replicates them with one ncclBroadcast per root instead of one per plane
        order = sorted(range(n), key=lambda i: (roots[i], i))
        for v in range(nvar):
            pool = torch.empty(sum(t.numel() for i in order for t in dev_frames[v][i]), dtype=torch.uint8, device=dev)
            off, packed = 0, {}
            for i in order:
                views = []
                for t in dev_frames[v][i]:
                    view = pool[off:off + t.numel()].view(t.shape)
                    view.copy_(t)
                    views.append(view)
                    off += t.numel()
                packed[i] = tuple(views)
            dev_frames[v] = [packed[i] for i in range(n)]
    dev_in = [in_array(dev_frames[v], F.MEM_DEVICE, lambda t: t.data_ptr()) for v in range(nvar)]
    comm_in, comm_roots = None, None
    if roots is not None:   # the exchange lists the frames root by root, so each root's pool is one contiguous run
        comm_roots = [roots[i] for i in order]
        comm_in = []
        for v in range(nvar):
            arr = (F.InputFrame * n)()
            for k, i in enumerate(order):
                C.memmove(C.byref(arr[k]), C.byref(dev_in[v][i]), C.sizeof(F.InputFrame))
            comm_in.append(arr)
    dev_out = (F.OutputFrame * n_out)()
    for k in range(n_out):
        dev_out[k].output_id = out_ids[k]
        dev_out[k].mem_kind = F.MEM_DEVICE
        dev_out[k].planes[0], dev_out[k].planes[1] = out_y[k].data_ptr(), out_uv[k].data_ptr()

    stream = torch.cuda.ExternalStream(r.cuda_stream(), device=dev)
    frame_ns = 33_333_333

    def step_dev(k):
        for a in dev_in[k % nvar]:
            a.pts_ns = k * frame_ns
        if roots is not None:   # the tick's exchange step: one NCCL group on the render stream
            r.comm_exchange_inputs(comm_in[k % nvar], n, comm_roots, None, pooled=True)
        r.render_raw(k * frame_ns, dev_in[k % nvar], n, dev_out, n_out, wait=False)

    # ---- value: device-resident, device-timed ---------------------------------------------------------
    # already streaming when the timed region starts (nvidia-smi takes ~0.2 s to start); rank 0 only -- its line is the
    # one that is printed, and N concurrent nvidia-smi loops would only contend for the driver lock
    # set-up, not warm-up: the first ticks of a handle compute the Lanczos weight tables, encode the TMA descriptors of
    # every frame buffer, size the arenas and take the clocks out of idle; the W warm-up steps follow
    t_setup = time.perf_counter()
    k = 0
    while k < 8 or time.perf_counter() - t_setup < SETUP_SECONDS:   # every GPU of the job reaches its load clocks (a rank whose
        step_dev(k % nvar)                                           # GPU ramps late would set the max over ranks)
        k += 1
        if k % 16 == 0:
            r.wait()
    r.wait()
    for k in range(args.warmup):
        step_dev(k)
    r.wait()
    barrier()
    clocks.mark()
    launches0 = r.stats()["kernel_launches"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.perf_counter()
    e0.record(stream)
    for k in range(args.steps):
        step_dev(args.warmup + k)
    t_submit = time.perf_counter() - t_wall0     # host time to plan and enqueue the ticks (GPU-bound when << the device time)
    r.wait()
    e1.record(stream)
    torch.cuda.synchronize()
    t_wall = time.perf_counter() - t_wall0
    barrier()
    ms = e0.elapsed_time(e1)
    launches = r.stats()["kernel_launches"] - launches0
    if args.dump_outputs:   # before the roofline and e2e legs below overwrite the output buffers
        prefix = f"rank{rank}_" if world > 1 else ""
        planes = {}
        for k in range(n_out):
            planes[f"{prefix}{out_ids[k].decode()}_y"] = out_y[k].cpu().numpy()
            planes[f"{prefix}{out_ids[k].decode()}_uv"] = out_uv[k].cpu().numpy()
        dump_outputs(args.dump_outputs, planes, DUMP_BYTES // world)
    ms_by_rank = [ms]
    if dist is not None:
        g = [torch.zeros(2, device=dev) for _ in range(world)]
        dist.all_gather(g, torch.tensor([ms, t_submit * 1e3], device=dev))
        ms_by_rank = [float(x[0].item()) for x in g]
        submit_by_rank = [float(x[1].item()) for x in g]
        ms = max(ms_by_rank)
    else:
        submit_by_rank = [t_submit * 1e3]
    clk = clocks.stop()
    ms_per_step = ms / args.steps
    value = world * n_out * args.steps / (ms * 1e-3)

    # ---- roofline: per-kernel device time from the library's own events -----------------------------
    r.set_profiling(True)
    for k in range(args.steps):
        step_dev(k)
        r.wait()
    kt = r.kernel_times()
    r.set_profiling(False)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    else:
        peak, peak_src = 6650.0, "B200_PROFILING.md fallback (of fallback)"
    per_kernel = {}
    for name, (tot, cnt) in kt.items():
        if cnt:
            per_launch_ms = tot / cnt
            launches_per_frame = cnt / args.steps
            per_kernel[name] = {"ms_per_launch": per_launch_ms, "launches_per_frame": launches_per_frame,
                                "ms_per_frame": tot / args.steps}
    dom = max(per_kernel, key=lambda k: per_kernel[k]["ms_per_frame"]) if per_kernel else None
    gpu_ms_frame = sum(v["ms_per_frame"] for v in per_kernel.values())
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")   # dram bytes per launch from the committed ncu capture
    if os.path.exists(tpath) and dom:
        traffic = json.load(open(tpath)).get(wl["name"], {}).get(dom)
    roofline = None
    if dom:
        # one launch of the dominant kernel processes one whole output frame's worth of its stage
        ach = wl["alg_bytes"] / (per_kernel[dom]["ms_per_frame"] * 1e-3) / 1e9
        roofline = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": traffic, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": wl["alg_bytes"] // max(1, round(per_kernel[dom]["launches_per_frame"])),
                    "kernel_share_of_gpu_time": per_kernel[dom]["ms_per_frame"] / gpu_ms_frame,
                    "whole_frame": {"achieved": wl["alg_bytes"] / (ms_per_step * 1e-3) / 1e9,
                                    "frac": wl["alg_bytes"] / (ms_per_step * 1e-3) / 1e9 / peak},
                    "kernels": per_kernel}

    # ---- e2e: through the C ABI with pinned HOST buffers --------------------------------------------------
    e2e = None
    if not args.no_e2e:
        hv = min(nvar, 2)
        host_frames = [[(dev_frames[v][i][0].cpu().pin_memory(), dev_frames[v][i][1].cpu().pin_memory())
                        for i in range(n)] for v in range(hv)]
        host_in = [in_array(host_frames[v], F.MEM_HOST, lambda t: t.data_ptr()) for v in range(hv)]
        # DEPTH sets of pinned output buffers: ticks k+1 and k+2 are submitted (smr_render_begin) before tick k is retired
        # (smr_render_end), so uploads, kernels and read-backs of neighbouring ticks overlap -- what the C ABI offers a caller
        DEPTH = 3
        hys = [[torch.empty((H, W), dtype=torch.uint8).pin_memory() for _ in range(n_out)] for _ in range(DEPTH)]
        huvs = [[torch.empty((H // 2, W // 2, 2), dtype=torch.uint8).pin_memory() for _ in range(n_out)] for _ in range(DEPTH)]
        host_out = []
        for b in range(DEPTH):
            arr = (F.OutputFrame * n_out)()
            for k in range(n_out):
                arr[k].output_id = out_ids[k]
                arr[k].mem_kind = F.MEM_HOST
                arr[k].planes[0], arr[k].planes[1] = hys[b][k].data_ptr(), huvs[b][k].data_ptr()
            host_out.append(arr)
        ke = max(5, min(args.steps, 200))   # enough ticks that one host hiccup cannot dominate sub-ms ticks
        def step_host(k, wait):
            for a in host_in[k % hv]:
                a.pts_ns = k * frame_ns          # fresh frames every tick (a frame older than the fallback timeout is dropped)
            r.render_raw(k * frame_ns, host_in[k % hv], n, host_out[k % DEPTH], n_out, wait=wait)
        for k in range(max(args.warmup, 8)):   # every in-flight slot (SMR_TICKS_IN_FLIGHT = 4) has its staging buffers allocated
            step_host(k, True)
        barrier()
        st0 = r.stats()
        ee0, ee1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        ee0.record(stream)
        acc = 0
        for k in range(ke):
            step_host(k, False)
            if k >= DEPTH - 1:
                r.wait()                                             # retires tick k - (DEPTH - 1)
                acc += int(hys[(k - DEPTH + 1) % DEPTH][0][0, 0])    # the step's result is read on the host
        for k in range(ke - DEPTH + 1, ke):
            r.wait()
            acc += int(hys[k % DEPTH][0][0, 0])
        ee1.record(stream)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        barrier()
        st1 = r.stats()
        e2e_s = max(wall, ee0.elapsed_time(ee1) * 1e-3)
        if dist is not None:
            t = torch.tensor([e2e_s], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_s = float(t.item())
        h2d_expected = n * iw * ih * 3 // 2
        assert (st1["h2d_bytes"] - st0["h2d_bytes"]) == h2d_expected * ke, "e2e leg: some ticks did not upload their inputs"
        h2d_step = (st1["h2d_bytes"] - st0["h2d_bytes"]) // ke
        d2h_step = (st1["d2h_bytes"] - st0["d2h_bytes"]) // ke
        # what the link can do on this box: pinned H2D of the same planes, back to back on one stream, nothing else running
        pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        probe_dst = [torch.empty_like(host_frames[0][i][0], device=dev) for i in range(n)]
        for rep in range(2):
            pe0.record()
            for i in range(n):
                probe_dst[i].copy_(host_frames[0][i][0], non_blocking=True)
            pe1.record()
            torch.cuda.synchronize()
        probe_gbs = sum(t.numel() for t in probe_dst) / (pe0.elapsed_time(pe1) * 1e-3) / 1e9
        fps_rank = n_out * ke / e2e_s
        e2e = {"value": world * n_out * ke / e2e_s, "unit": "frames/s", "steps": ke,
               "h2d_bytes_per_step": h2d_step, "d2h_bytes_per_step": d2h_step,
               "pcie_h2d_gbs": h2d_step * (ke / e2e_s) / 1e9, "pcie_d2h_gbs": d2h_step * (ke / e2e_s) / 1e9,
               "pcie_h2d_probe_gbs": probe_gbs, "pcie_frac_of_probe": h2d_step * (ke / e2e_s) / 1e9 / probe_gbs,
               "per_gpu_frames_s": fps_rank}

    # ---- cpu baseline (rank 0, N = 1 only) ------------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        times, desc, cores = cpu_steps(wl, 5, 1)   # the same procedure as the --impl reference arm
        cpu = {"value": 1.0 / float(np.median(times)), "unit": "frames/s", "cores": cores, "kind": "port", "sample": desc,
               "spread": {"min_ms": float(np.min(times)) * 1e3, "max_ms": float(np.max(times)) * 1e3, "steps": len(times)}}

    secondary = None
    if world > 1 and wl["name"] == "cfg3" and not args.no_secondary:
        modes = ["nccl", "peer_copy", "peer_direct"] if args.exchange == "all" else [args.exchange]
        try:
            secondary = measure_cfg4_modes(torch, dist, dev, rank, world, local, max(args.steps, 20), args.warmup, modes)
        except Exception as e:   # the primary line stands on its own; say what happened to the exchange leg
            secondary = {"workload": "cfg4", "error": repr(e)[:300]}
    if rank == 0:
        line = {"metric": metric_name(wl),
                "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32 math on u8 planes (f16 resampler scratch)", "data": "synthetic",
                "config": {"workload": wl["name"], "detail": wl["desc"], "outputs_per_gpu": n_out,
                           "nvlink_broadcast_bytes_per_tick": (n * iw * ih * 3 // 2) * (world - 1) if roots is not None else (secondary or {}).get("nvlink_broadcast_bytes_per_tick", 0),
                           "l2_policy": f"inputs larger than L2: {nvar} distinct frame sets of "
                                        f"{wl['alg_bytes'] / 1e6:.0f} MB cycled (> 126 MB L2)",
                           "algorithmic_bytes_per_frame": wl["alg_bytes"], "wall_s_timed_region": t_wall,
                           "device_ms_per_step_by_rank": [m / args.steps for m in ms_by_rank],
                           "host_submit_ms_per_step_by_rank": [m / args.steps for m in submit_by_rank],
                           "secondary": secondary},
                "clocks": clk, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu}
        print(json.dumps(line))
    if roots is not None:
        r.comm_destroy()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
