#!/usr/bin/env python
"""bench.py -- headline benchmark of the DMesh tile rasterizer hot path on B200.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload C4|C2|C1|C5]
                    [--views-per-call V] [--no-per-config] [--dump-outputs DIR]

Metric (BASELINE.json): fwd+bwd throughput in views/s (and ms per 1024x1024 view) of the tri renderer, at
1/2/4/8 B200, next to the reference CUDA extension on the same box.

Default workload = BASELINE.json configs[3] ("C4"): the multi-view DMesh optimisation step -- 1 M triangles,
64 views at 1024x1024, cameras sharded over the N ranks (STRONG scaling: the job is always the same 64 views; rank r
renders views r*64/N .. (r+1)*64/N - 1 in calls of --views-per-call views), followed by ONE all-reduce of the packed
per-triangle / per-vertex scene gradients.  A "step" = that whole optimisation step through the PUBLIC API
(TriRenderer -> autograd -> _C shim -> C ABI -> sm_100a kernels; dmesh_renderer_b200/multiview.py for the sharding
and the collective).  `value` = 64 views / step time with the step inputs resident in HBM; `e2e` = the same step
with the per-step host inputs (cameras and target images, pinned host memory) copied H2D inside the timed region and
the scalar loss read back D2H.

--impl reference: the UNMODIFIED reference CUDA extension (oracle/_ref, built from /root/reference by
oracle/build_ref.py) runs the same job with the same protocol: every rank renders its 64/N views through
_C.render_tris / render_tris_backward exactly as the reference's Python wrapper calls them, then torch.distributed
all-reduces the three view-summed gradient tensors (BASELINE.md section 3a).  The reference has no CPU
implementation; the CPU oracle (oracle/oracle.cpp) is timed as `cpu_baseline` on our arm's line and is the fallback
of the reference arm when oracle/_ref cannot be loaded.

At N = 1 both arms also time the other BASELINE configs at the `_C` level (`per_config`: C1, C2, C5 tri; C3 tet),
so that every ours-vs-reference ratio quoted in README.md is a driver-run number.

--dump-outputs DIR (our arm): after the timed steps, write what the last timed step computed for rank 0 -- the
gradients the step leaves in the scene leaves (all-reduced) and in the per-call verts_depth / faces_intense leaves,
and the colour and depth images of every call -- as DIR/<name>.npy (float32).  An array of more than DUMP_SAMPLE
elements is stored as a fixed sample of it: the flattened array at sorted indices drawn by
torch.randint(0, numel, (DUMP_SAMPLE,)) from a CPU generator seeded with 0.  The inputs are seeded, so two builds
run with the same arguments can be compared output for output.  The last timed step keeps its images alive (about
1 GB at C4 on one GPU) until they are written, so the timings of a dumping run are not the headline numbers.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

METRIC = "tri_fwd_bwd_views_per_sec_1024x1024"
UNIT = "views/s"
TOTAL_VIEWS_C4 = 64
DUMP_SAMPLE = 1 << 21     # elements kept per dumped array: 7 arrays x 8 MB stay under 64 MB


# --------------------------------------------------------------------------- helpers
def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


class L2Flush:
    """Write a buffer larger than the 126 MB L2 between timed steps."""

    def __init__(self, device, mbytes=256):
        self.buf = torch.empty(mbytes * 1024 * 1024, dtype=torch.uint8, device=device)
        self.v = 0

    def __call__(self):
        self.v = (self.v + 1) & 0xff
        self.buf.fill_(self.v)


CPU_BINDING = None   # cores this rank was bound to (N > 1 only)


def dist_setup(gpus):
    ws = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if ws > 1:
        torch.cuda.set_device(local)
        if os.environ.get("DMR_BENCH_NO_CPU_BINDING") != "1":
            from dmesh_renderer_b200.multiview import bind_to_gpu_cpus
            cores = bind_to_gpu_cpus(local)     # pinned staging buffers on the GPU's own NUMA node
            global CPU_BINDING
            CPU_BINDING = len(cores) if cores else None
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(0)
    return ws, rank, local


def barrier(ws):
    if ws > 1:
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(x, ws, dev):
    if ws == 1:
        return x
    t = torch.tensor([x], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def bit_length(n):
    return max(int(n).bit_length(), 1)


def dump_outputs(out_dir, arrays):
    """Write each device tensor as out_dir/<name>.npy (float32): whole, or a flat seeded sample if it is large
    (module doc)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_SAMPLE:
            idx = torch.randint(0, t.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0))
            t = t.reshape(-1)[idx.sort().values.to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


# --------------------------------------------------------------------------- workload
class Workload:
    """Scene replicated on every rank (device) + this rank's views split into calls + pinned host copies of the
    per-step host inputs (cameras, target images)."""

    def __init__(self, name, rank, ws, dev, views_per_call):
        from dmesh_renderer_b200 import scenes
        from dmesh_renderer_b200.multiview import shard_views
        self.name = name
        if name == "C4":     # 64 views sharded over the ranks (strong scaling)
            mine = shard_views(TOTAL_VIEWS_C4, rank, ws)
            base = scenes.config("C4", views=TOTAL_VIEWS_C4, view_slice=slice(mine.start, mine.stop))
            self.total_views, self.scaling = TOTAL_VIEWS_C4, "strong"
        elif name in ("C1", "C2", "C5"):   # one view per rank (weak scaling): camera r of a seeded ring around the scene
            base = scenes.config(name)
            if ws > 1:
                g = torch.Generator().manual_seed(99)
                dirs = scenes.fibonacci_dirs(max(ws, 2), g)
                mv, pj = scenes.cameras(dirs[rank:rank + 1], 3.0, base.W, base.H, 0.5, 6.0)
                base = base._replace(mv_mats=mv, proj_mats=pj, verts_depth=scenes.ndc_depth(base.verts, mv, pj))
            self.total_views, self.scaling = ws, "weak"
        else:
            raise SystemExit("unknown workload " + name)
        self.local_views = base.mv_mats.shape[0]
        self.vpc = max(1, min(views_per_call or self.local_views, self.local_views))
        self.s = scenes.to_device(base, dev)
        self.H, self.W = base.H, base.W
        gen = torch.Generator().manual_seed(1234 + rank)
        B = self.local_views
        self.host = {"mv": base.mv_mats.contiguous().pin_memory(), "proj": base.proj_mats.contiguous().pin_memory(),
                     "target_color": torch.rand(B, 3, base.H, base.W, generator=gen).pin_memory(),
                     "target_depth": torch.rand(B, 1, base.H, base.W, generator=gen).pin_memory()}
        self.calls = [(a, min(B, a + self.vpc)) for a in range(0, B, self.vpc)]

    def describe(self, ws):
        s = self.s
        cfgname = {"C1": "configs[0]", "C2": "configs[1]", "C4": "configs[3]", "C5": "configs[4]"}[self.name]
        if self.name == "C4":
            what = ("%s: multi-view DMesh optimisation step, tri renderer fwd+bwd, %d triangles, %d views at %dx%d sharded "
                    "over %d GPU(s) = %d views per rank in calls of %d, one all-reduce of the (6P+F) fp32 scene gradients"
                    % (cfgname, s.faces.shape[0], self.total_views, s.W, s.H, ws, self.local_views, self.vpc))
        else:
            what = "%s: tri renderer fwd+bwd, %d triangles, %dx%d, 1 view per rank and step" % (cfgname, s.faces.shape[0], s.W, s.H)
        return {"workload": what, "triangles": int(s.faces.shape[0]), "vertices": int(s.verts.shape[0]), "image": [s.H, s.W],
                "views_per_step_total": self.total_views, "views_per_rank": self.local_views, "views_per_call": self.vpc,
                "parallelism": ("cameras sharded x%d, scene replicated" % ws) if ws > 1 else "single GPU",
                "l2_flush": "256 MB device fill between timed steps, outside the timed events",
                "e2e_host_inputs": "cameras + target colour/depth images of this rank's views (pinned host memory, copied per "
                                   "call on a copy stream that runs one call ahead" +
                                   (", across step boundaries too: the K timed steps run back to back in one region, per-step "
                                    "working set >> L2" if self.name == "C4" else "; one timed region per step, L2 flushed in between") +
                                   "); verts_depth / faces_intense are scene-derived device tensors (DMesh computes them from "
                                   "the scene on the GPU), the scene is resident",
                "e2e_result_read": "the scalar image loss of every step is copied D2H into pinned memory and read by the "
                                   "host (stream synchronisation) before the next step is enqueued"}


# --------------------------------------------------------------------------- our arm
def run_ours(args, ws, rank, local):
    from dmesh_renderer_b200 import TriRenderer, TriRenderSettings, _lib
    from dmesh_renderer_b200.multiview import PackedSceneGrads
    dev = torch.device("cuda", local)
    wl = Workload(args.workload, rank, ws, dev, args.views_per_call)
    s = wl.s
    lib = _lib.load()
    renderer = TriRenderer(TriRenderSettings(s.H, s.W, s.bg))
    leaves = PackedSceneGrads(s.verts.clone(), s.verts_color.clone(), s.faces_opacity.clone())
    verts, vcol, fopa = leaves.leaves
    # per-call leaf tensors of the per-view inputs (their gradients stay rank-local)
    vdep = [s.verts_depth[a:b].clone().requires_grad_() for a, b in wl.calls]
    fint = [s.faces_intense[a:b].clone().requires_grad_() for a, b in wl.calls]
    mvs = [s.mv_mats[a:b].contiguous() for a, b in wl.calls]
    pjs = [s.proj_mats[a:b].contiguous() for a, b in wl.calls]
    tgt_c = [wl.host["target_color"][a:b].to(dev) for a, b in wl.calls]
    tgt_d = [wl.host["target_depth"][a:b].to(dev) for a, b in wl.calls]
    flush = L2Flush(dev)
    images = [None] * len(wl.calls)     # --dump-outputs: the images of the last timed step, per call

    def step_device(keep_images=False):
        leaves.zero_()
        with leaves.direct():   # backward kernels accumulate straight into the packed gradient buffer
            for i in range(len(wl.calls)):
                vdep[i].grad = None
                fint[i].grad = None
                color, depth = renderer(verts, s.faces, vcol, fopa, mvs[i], pjs[i], vdep[i], fint[i])
                if keep_images:
                    images[i] = (color.detach(), depth.detach())
                # gradient of the image loss 0.5 * ||render - target||^2 as cotangent (device resident targets)
                torch.autograd.backward([color, depth], [color.detach() - tgt_c[i], depth.detach() - tgt_d[i]])
        leaves.all_reduce()

    # ---- e2e: cameras + targets of call i+1 travel H2D on a copy stream while call i renders (two staging slots)
    copy_stream = torch.cuda.Stream(device=dev)
    nslot = 2
    stage = [{"mv": torch.empty_like(mvs[0]), "proj": torch.empty_like(pjs[0]), "tc": torch.empty_like(tgt_c[0]),
              "td": torch.empty_like(tgt_d[0]), "cams": None, "ready": None, "free": None} for _ in range(nslot)]
    loss_acc = torch.zeros(1, device=dev)
    loss_host = torch.zeros(1).pin_memory()
    h2d_bytes = sum(v.numel() * v.element_size() for v in wl.host.values())

    ncalls = len(wl.calls)

    def enqueue_copy(c):
        """H2D of the inputs of global call number c (step c // ncalls, call c % ncalls) into staging slot c % nslot."""
        a, b = wl.calls[c % ncalls]
        st = stage[c % nslot]
        n = b - a
        if st["free"] is not None:
            copy_stream.wait_event(st["free"])      # the call that last used this slot has consumed it
        with torch.cuda.stream(copy_stream):
            st["mv"][:n].copy_(wl.host["mv"][a:b], non_blocking=True)
            st["proj"][:n].copy_(wl.host["proj"][a:b], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
            st["cams"] = ev                         # the forward pass needs only the cameras; the targets follow
            st["tc"][:n].copy_(wl.host["target_color"][a:b], non_blocking=True)
            st["td"][:n].copy_(wl.host["target_depth"][a:b], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
            st["ready"] = ev

    def e2e_begin():
        main = torch.cuda.current_stream()
        for st in stage:
            st["free"] = None
        copy_stream.wait_stream(main)               # earlier readers of the staging slots are done
        enqueue_copy(0)

    def step_e2e(k, last_step):
        """Step k of an e2e region opened by e2e_begin().  The copy stream runs ONE CALL AHEAD of the compute stream,
        across step boundaries too (a data loader that prefetches the next batch): every step's inputs are copied
        inside the region, once per step."""
        main = torch.cuda.current_stream()
        leaves.zero_()
        loss_acc.zero_()
        with leaves.direct():
            for i, (a, b) in enumerate(wl.calls):
                c = k * ncalls + i
                if i + 1 < ncalls or not last_step:
                    enqueue_copy(c + 1)
                st, n = stage[c % nslot], b - a
                main.wait_event(st["cams"])
                vdep[i].grad = None
                fint[i].grad = None
                color, depth = renderer(verts, s.faces, vcol, fopa, st["mv"][:n], st["proj"][:n], vdep[i], fint[i])
                main.wait_event(st["ready"])        # target images: they travelled while the forward pass ran
                dc, dd = color.detach() - st["tc"][:n], depth.detach() - st["td"][:n]
                torch.autograd.backward([color, depth], [dc, dd])
                # 0.5 * ||render - target||^2: one reduction pass per image stack (no squared temporaries)
                loss_acc.add_(0.5 * (torch.linalg.vector_norm(dc).square() + torch.linalg.vector_norm(dd).square()))
                ev = torch.cuda.Event()
                ev.record(main)
                st["free"] = ev
        leaves.all_reduce()
        loss_host.copy_(loss_acc, non_blocking=True)
        main.synchronize()                          # the step's result is read on the host every step
        return float(loss_host[0])

    # ---- warm-up
    for _ in range(max(args.warmup, 3)):
        step_device()
    barrier(ws)

    # ---- which collective runs, and is it right?  (outside the timed regions)
    collective = None
    if ws > 1:
        g = torch.Generator(device=dev).manual_seed(77 + rank)
        x = torch.randn(leaves.flat.numel(), device=dev, generator=g)
        ref = x.clone()
        dist.all_reduce(ref)
        leaves.flat.copy_(x)
        leaves.all_reduce()
        torch.cuda.synchronize()
        same = bool(torch.equal(leaves.flat, ref))
        rel = float(((leaves.flat - ref).norm() / ref.norm()).item())
        ok = torch.tensor([1 if same else 0, 1 if rel < 1e-6 else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        collective = {"path": "nvls" if leaves.collective == "nvls" else "nccl", "detail": leaves.collective,
                      "check": "bit-identical to torch.distributed.all_reduce (NCCL) on every rank" if int(ok[0]) else
                               ("rel L2 %.2e vs NCCL" % rel if int(ok[1]) else "MISMATCH vs NCCL: rel L2 %.2e" % rel),
                      "floats": int(leaves.flat.numel())}
        leaves.zero_()

    # ---- timed region 1: device-resident inputs, CUDA events per step, L2 flushed between steps
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = lib.dmr_launch_count()
    total_ms = 0.0
    for k in range(args.steps):
        flush()
        barrier(ws)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        step_device(keep_images=bool(args.dump_outputs) and k == args.steps - 1)
        b.record()
        barrier(ws)
        total_ms += a.elapsed_time(b)
    launches = int(lib.dmr_launch_count() - launches0)
    total_ms = max_over_ranks(total_ms, ws, dev)
    clocks = sampler.stop() if rank == 0 else None
    ms_per_step = total_ms / args.steps
    value = wl.total_views / (ms_per_step / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {
            "grad_verts": verts.grad, "grad_verts_color": vcol.grad, "grad_faces_opacity": fopa.grad,
            "grad_verts_depth": torch.cat([t.grad for t in vdep]), "grad_faces_intense": torch.cat([t.grad for t in fint]),
            "color": torch.cat([c for c, _ in images]), "depth": torch.cat([d for _, d in images])})

    # ---- timed region 2: per-kernel durations (stage events inside the library, on the launching stream) for the
    #      roofline: one step, read after every call (a stage's events are overwritten by the next call)
    nst = lib.dmr_profile_stage_count()
    names = [lib.dmr_profile_stage_name(i).decode() for i in range(nst)]
    acc, cnt = [0.0] * nst, [0] * nst
    buf = (ctypes.c_float * nst)()

    def read_stages():
        lib.dmr_profile_read(buf)
        for i in range(nst):
            if buf[i] >= 0:
                acc[i] += buf[i]
                cnt[i] += 1
    lib.dmr_profile_enable(1)
    nprof = min(args.steps, 5)
    for _ in range(nprof):
        flush()
        torch.cuda.synchronize()
        leaves.zero_()
        for i in range(len(wl.calls)):
            vdep[i].grad = None
            fint[i].grad = None
            color, depth = renderer(verts, s.faces, vcol, fopa, mvs[i], pjs[i], vdep[i], fint[i])
            read_stages()
            torch.autograd.backward([color, depth], [color.detach() - tgt_c[i], depth.detach() - tgt_d[i]])
            read_stages()
    lib.dmr_profile_enable(0)
    stage_ms = {names[i]: acc[i] / cnt[i] for i in range(nst) if cnt[i]}      # per launch (= per call of vpc views)
    stats = scene_stats(s, mvs[0], pjs[0], vdep[0].detach(), fint[0].detach())

    # ---- timed region 3: end to end (host inputs, H2D + D2H inside), wall clock.
    #      C4: the K steps run back to back in ONE region (the working set of a step -- >= 1.4 GB of state buffers per
    #      call -- is far larger than the 126 MB L2, so no flush is needed between them) and the copy stream prefetches
    #      the next call's inputs across step boundaries; all K x h2d_bytes_per_step are copied inside the region.
    #      Small workloads (C1, C2, C5: one call per step, working set comparable to L2): one region per step with the
    #      L2 flushed in between, no prefetch across steps.
    pipelined = wl.name == "C4"
    e2e_begin()
    for k in range(2):
        step_e2e(k, k == 1)
    e2e_s = 0.0
    if pipelined:
        barrier(ws)
        t0 = time.perf_counter()
        e2e_begin()
        for k in range(args.steps):
            step_e2e(k, k == args.steps - 1)
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
    else:
        for _ in range(args.steps):
            flush()
            barrier(ws)
            t0 = time.perf_counter()
            e2e_begin()
            step_e2e(0, True)
            torch.cuda.synchronize()
            e2e_s += time.perf_counter() - t0
    e2e_s = max_over_ranks(e2e_s, ws, dev)
    e2e_value = wl.total_views / (e2e_s / args.steps)

    per_config = None
    if ws == 1 and not args.no_per_config:
        del tgt_c, tgt_d, stage
        torch.cuda.empty_cache()
        per_config = per_config_times("ours", dev)

    if rank != 0:
        return
    # ---- roofline of the dominant kernel.  Algorithmic bytes per LAUNCH (one call = vpc views of this rank):
    #      SURVEY.md 8d / DESIGN.md 3 per-unit figures x the units of one launch.
    P, F, px, vpc = int(s.verts.shape[0]), int(s.faces.shape[0]), s.H * s.W, wl.vpc
    R = stats["instances_R_per_call"]
    tiles = vpc * ((s.W + 15) // 16) * ((s.H + 15) // 16)
    npass = (bit_length(tiles) + 7) // 8          # instance sort: tile bits only (two-level binning, DESIGN.md 3.1)
    BF = F * vpc
    alg = {
        # positions / indices / colours / opacity are read once per call (the kernels walk the views inside a thread)
        "preprocess_points": 12 * P + 20 * P * vpc, "preprocess_faces": (12 + 72 + 4) * F + (48 + 4 + 16 + 144) * BF,
        "face_depth_sort": (4 + 4 * 16) * BF,      # histogram read + 4 eight-bit passes over (u32 key, u32 index) pairs
        "scan": 12 * BF,                           # order + gathered tiles_touched read, offsets written
        "duplicate_with_keys": 16 * BF + 8 * R,    # order, offsets, rect read; (u32 tile, u32 face) written
        "sort_histogram": 4 * R,
        "tile_ranges": 4 * R + 8 * tiles,
        "tri_render_forward": 132 * R + 28 * px * vpc,
        "tri_render_backward": 132 * R + 28 * px * vpc + 4 * (6 * P + F) + 4 * (P + F) * vpc,
        # statistics of every (view, face); the triangle (96 B of the record) and the vertex scatter once per face
        "tri_grad_finish": 96 * BF + 96 * F + 4 * (6 * P + F) + 4 * (P + F) * vpc,
    }
    for i in range(8):
        alg["sort_pass%d" % i] = 16 * R
    dom = max(stage_ms, key=stage_ms.get)
    peak, peak_src = peaks()
    achieved = alg.get(dom, 0) / (stage_ms[dom] * 1e-3) / 1e9
    traffic, winst, tsrc = None, None, None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        with open(tp) as f:
            tj = json.load(f)
        ent = tj.get(args.workload, {}).get(dom)
        if isinstance(ent, dict):
            # per launch of the captured configuration, scaled to this launch's views where the capture had fewer
            scale = vpc / float(ent.get("views", vpc))
            traffic = int(ent["dram_bytes"] * scale)
            winst = int(ent["warp_instructions"] * scale)
            tsrc = ent.get("source")
    hbm_stages = {k: round(alg[k] / (v * 1e-3) / 1e9 / peak, 3) for k, v in stage_ms.items()
                  if k in alg and not k.startswith("tri_render")}
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    roofline = {"kernel": dom, "bound": "hbm", "achieved": round(achieved, 2), "peak": peak, "unit": "GB/s",
                "frac": round(achieved / peak, 4), "traffic": traffic, "traffic_source": tsrc, "peak_source": peak_src,
                "kernel_ms": round(stage_ms[dom], 4), "algorithmic_bytes": alg.get(dom, 0),
                "per_launch": "one call = %d view(s) of this rank" % vpc,
                "note": "render kernels are issue-bound (coverage tests + shading), not HBM-bound; see DESIGN.md",
                "stage_ms": {k: round(v, 4) for k, v in stage_ms.items()}, "instances_R_per_call": R, "sort_passes": npass,
                "hbm_frac_of_streaming_stages": hbm_stages}
    if winst:
        # the bound that actually limits the dominant kernel: warp-instruction issue (148 SMs x 4 schedulers x SM clock);
        # instruction count from the tracked ncu capture named in traffic_source, duration measured live above
        peak_issue = 148 * 4 * sm_mhz * 1e6
        roofline["issue_bound"] = {"warp_instructions": winst, "achieved_ginst_per_s": round(winst / (stage_ms[dom] * 1e-3) / 1e9, 1),
                                   "peak_ginst_per_s": round(peak_issue / 1e9, 1),
                                   "frac": round(winst / (stage_ms[dom] * 1e-3) / peak_issue, 3)}
    # compute-side figure of the render kernels (SURVEY.md 8d): pixel x instance pair tests against the ~4.6 T tests/s
    # bound (148 SMs x 128 lanes x SM clock / ~8 lane-ops per test)
    if stats.get("pair_tests_per_view") and "tri_render_forward" in stage_ms:
        bound = 148 * 128 * sm_mhz * 1e6 / 8.0
        pt = stats["pair_tests_per_view"] * vpc
        roofline["pair_tests"] = {"per_view": stats["pair_tests_per_view"], "definition": "sum over tiles of 256 x instances traversed before tile-wide termination",
                                  "forward_tests_per_s": round(pt / (stage_ms["tri_render_forward"] * 1e-3), 0),
                                  "bound_tests_per_s": round(bound, 0),
                                  "forward_frac": round(pt / (stage_ms["tri_render_forward"] * 1e-3) / bound, 4)}

    cpu = cpu_baseline(args.workload) if ws == 1 else None
    out = {"metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": ws, "steps": args.steps,
           "warmup": max(args.warmup, 3), "ms_per_step": round(ms_per_step, 4), "higher_is_better": True,
           "scaling": wl.scaling, "vs_baseline": None, "dtype": "f32",
           "data": "synthetic (seeded, SURVEY.md App. E)", "config": wl.describe(ws),
           "ms_per_view": round(ms_per_step / wl.local_views, 4),
           "e2e": {"value": round(e2e_value, 3), "unit": UNIT, "h2d_bytes_per_step": int(h2d_bytes),
                   "d2h_bytes_per_step": 4, "ms_per_step": round(e2e_s / args.steps * 1e3, 4)},
           "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "impl": "dmesh_renderer_b200",
           "scene_stats": stats}
    if collective:
        out["collective"] = collective
    if ws > 1:
        out["config"]["host_cores_bound_to_gpu_numa_node"] = CPU_BINDING
    if per_config:
        out["per_config"] = per_config
    if cpu:
        out["cpu_baseline"] = cpu
    print(json.dumps(out), flush=True)


def scene_stats(s, mv, pj, vdep, fint):
    """R and the pair-test count of one call of the workload (SURVEY.md 8d 'compute-side figure for render')."""
    from dmesh_renderer_b200 import _C, debug
    mvt, pjt = mv.transpose(1, 2), pj.transpose(1, 2)
    R, _, _, pb, fb, bb, ib = _C.render_tris(s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mvt, pjt,
                                             torch.inverse(mvt), torch.inverse(pjt), vdep, fint, s.H, s.W)
    B, P, F = mv.shape[0], s.verts.shape[0], s.faces.shape[0]
    out = {"instances_R_per_call": int(R), "views_in_call": int(B)}
    try:
        dims = dict(B=B, P=P, F=F, W=s.W, H=s.H, R=R)
        ranges = debug.view_torch("tri", "ranges", ib, **dims).to(torch.int64)
        ncon = debug.view_torch("tri", "n_contrib", ib, **dims).to(torch.int64).view(B, s.H, s.W)
        fT = debug.view_torch("tri", "final_T", ib, **dims).view(B, s.H, s.W)
        tx, ty = (s.W + 15) // 16, (s.H + 15) // 16
        if s.W % 16 == 0 and s.H % 16 == 0:
            total = (ranges[:, 1] - ranges[:, 0]).view(B, ty, tx)
            nc = ncon.view(B, ty, 16, tx, 16).amax(dim=(2, 4))
            alive = (fT >= 1e-4).view(B, ty, 16, tx, 16).any(dim=4).any(dim=2)   # some pixel never terminated: whole list walked
            trav = torch.where(alive, total, nc)
            out["pair_tests_per_view"] = int((trav.sum() * 256 // B).item())
            out["instances_traversed_per_view"] = int((trav.sum() // B).item())
            out["hits_per_pixel_mean"] = None
    except Exception as ex:   # statistics only
        out["pair_tests_error"] = repr(ex)
    return out


def cpu_baseline(workload):
    """The CPU oracle (oracle/oracle.cpp, OpenMP) on the host cores: fwd+bwd of one view of the workload."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    try:
        import oracle
        from dmesh_renderer_b200 import scenes
        if workload == "C4":
            s, name = scenes.config("C4", views=1), "C4 (1 of its 64 views)"
        else:
            name = workload if workload in ("C1", "C2") else "C2"
            s = scenes.config(name)
        gc, gd = scenes.cotangents(s)
        t0 = time.perf_counter()
        o = oracle.TriOracle(s)
        o.backward(gc, gd)
        dt = time.perf_counter() - t0
        o.close()
        return {"value": round(1.0 / dt, 4), "unit": UNIT, "cores": oracle.num_threads(), "kind": "port",
                "sample": "1 full fwd+bwd view of %s (%d triangles, %dx%d), %.2f s" % (name, s.faces.shape[0], s.W, s.H, dt)}
    except Exception as ex:   # the oracle is a reported baseline only
        return {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "unavailable: %r" % (ex,)}


# --------------------------------------------------------------------------- the other BASELINE configs, _C level
def per_config_times(impl, dev, n=15, warm=4):
    """fwd / bwd / fwd+bwd ms (median, CUDA events) of C1, C2, C5 (tri) and C3 (tet) through the four `_C` entry
    points -- the same calls, same seeded scenes and same protocol in both arms (tools/time_compare.py)."""
    from dmesh_renderer_b200 import scenes
    if impl == "ours":
        from dmesh_renderer_b200 import _C as C
    else:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import build_ref
        C = build_ref.load()

    def timeit(fn):
        for _ in range(warm):
            fn()
        ts = []
        for _ in range(n):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        ts.sort()
        return round(ts[len(ts) // 2], 4)

    out = {}
    for name in ("C1", "C2", "C5", "C3"):
        try:
            cpu = scenes.config(name)
            s = scenes.to_device(cpu, dev)
            gc, gd = [t.to(dev) for t in scenes.cotangents(cpu)]
            mv, pj = s.mv_mats.transpose(1, 2).contiguous(), s.proj_mats.transpose(1, 2).contiguous()
            imv, ipj = torch.inverse(mv), torch.inverse(pj)
            st = {}
            if s.kind == "tri":
                fa = (s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, imv, ipj, s.verts_depth, s.faces_intense)

                def fwd():
                    st["o"] = C.render_tris(*fa, s.H, s.W)

                def bwd():
                    o = st["o"]
                    C.render_tris_backward(*fa, gc, gd, o[0], o[3], o[4], o[5], o[6])
            else:
                fa = (s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mv, pj, imv, ipj, s.verts_depth,
                      s.faces_intense, s.tets, s.face_tets, s.tet_faces)

                def fwd():
                    st["o"] = C.render_tets(*fa, s.H, s.W, 0)

                def bwd():
                    o = st["o"]
                    C.render_tets_backward(*fa, gc, gd, o[3], o[4], o[5], o[6])

            def both():
                fwd()
                bwd()
            e = {"ms_fwd": timeit(fwd), "ms_bwd": timeit(bwd), "ms_fwd_bwd": timeit(both),
                 "image": [s.H, s.W], "faces": int(s.faces.shape[0])}
            if s.kind == "tri":
                e["R"] = int(st["o"][0])
            e["ms_fwd_bwd_per_1024x1024"] = round(e["ms_fwd_bwd"] * 1024 * 1024 / (s.H * s.W), 4)
            out[name] = e
            del s, gc, gd, st
            torch.cuda.empty_cache()
        except Exception as ex:
            out[name] = {"error": repr(ex)}
    out["protocol"] = "median of %d after %d warm-ups, CUDA events, `_C` entry points (no autograd), seeded scenes of SURVEY.md App. E" % (n, warm)
    return out


# --------------------------------------------------------------------------- reference arm
def run_reference(args, ws, rank, local):
    dev = torch.device("cuda", local)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import build_ref
    ref = None
    try:
        ref = build_ref.load()
    except Exception as ex:
        sys.stderr.write("reference extension failed to load: %r\n" % (ex,))
    if ref is None:
        if rank != 0:
            return
        wl = Workload(args.workload, 0, 1, dev, args.views_per_call)
        cpu = cpu_baseline(args.workload)
        out = {"metric": METRIC, "value": cpu["value"], "unit": UNIT, "n_gpus": ws, "steps": 1, "warmup": 0,
               "ms_per_step": round(1e3 / cpu["value"], 3) if cpu["value"] else None, "higher_is_better": True,
               "scaling": wl.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": wl.describe(1),
               "impl": "reference", "cpu_baseline": cpu,
               "e2e": {"value": cpu["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
               "note": "oracle/_ref (the reference CUDA extension) could not be loaded; CPU oracle port timed instead"}
        print(json.dumps(out), flush=True)
        return
    wl = Workload(args.workload, rank, ws, dev, args.views_per_call)
    s = wl.s
    mvs = [s.mv_mats[a:b].transpose(1, 2).contiguous() for a, b in wl.calls]
    pjs = [s.proj_mats[a:b].transpose(1, 2).contiguous() for a, b in wl.calls]
    vdep = [s.verts_depth[a:b].contiguous() for a, b in wl.calls]
    fint = [s.faces_intense[a:b].contiguous() for a, b in wl.calls]
    tgt_c = [wl.host["target_color"][a:b].to(dev) for a, b in wl.calls]
    tgt_d = [wl.host["target_depth"][a:b].to(dev) for a, b in wl.calls]
    flush = L2Flush(dev)
    P, F = s.verts.shape[0], s.faces.shape[0]
    packed = torch.zeros(6 * P + F, device=dev)       # [dL_dverts | dL_dvcolor | dL_dfopacity], one all-reduce
    gv, gcol, gop = packed[:3 * P].view(P, 3), packed[3 * P:6 * P].view(P, 3), packed[6 * P:]

    def step():
        packed.zero_()
        for i in range(len(wl.calls)):
            # exactly what the reference's Python wrapper does per call (reference __init__.py:62-88, 124-149)
            imv, ipj = torch.inverse(mvs[i]), torch.inverse(pjs[i])
            a = (s.bg, s.verts, s.faces, s.verts_color, s.faces_opacity, mvs[i], pjs[i], imv, ipj, vdep[i], fint[i])
            R, color, depth, pb, fb, bb, ib = ref.render_tris(*a, s.H, s.W)
            g = ref.render_tris_backward(*a, color - tgt_c[i], depth - tgt_d[i], R, pb, fb, bb, ib)
            if len(wl.calls) == 1 and ws == 1:
                continue                                  # single call, single GPU: the returned tensors ARE the result
            gv.add_(g[0])
            gcol.add_(g[1])
            gop.add_(g[2])
        if ws > 1:
            dist.all_reduce(packed)                       # BASELINE.md 3a: torch NCCL all-reduce of the view-summed grads

    for _ in range(max(args.warmup, 3)):
        step()
    barrier(ws)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    total_ms = 0.0
    for _ in range(args.steps):
        flush()
        barrier(ws)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        step()
        b.record()
        barrier(ws)
        total_ms += a.elapsed_time(b)
    total_ms = max_over_ranks(total_ms, ws, dev)
    clocks = sampler.stop() if rank == 0 else None
    ms = total_ms / args.steps
    value = wl.total_views / (ms / 1e3)
    per_config = None
    if ws == 1 and not args.no_per_config:
        del tgt_c, tgt_d
        torch.cuda.empty_cache()
        per_config = per_config_times("reference", dev)
    if rank != 0:
        return
    out = {"metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": ws, "ranks_used": ws, "steps": args.steps,
           "warmup": max(args.warmup, 3), "ms_per_step": round(ms, 4), "higher_is_better": True, "scaling": wl.scaling,
           "vs_baseline": None, "dtype": "f32", "data": "synthetic (seeded, SURVEY.md App. E)", "config": wl.describe(ws),
           "ms_per_view": round(ms / wl.local_views, 4), "impl": "reference", "clocks": clocks,
           "note": "the reference has no multi-GPU path: every rank runs its unmodified CUDA extension on its share of the views "
                   "and torch.distributed all-reduces the three view-summed gradient tensors (BASELINE.md 3a)",
           "cpu_baseline": {"value": round(value, 3), "unit": UNIT, "cores": 1, "kind": "reference",
                            "sample": "the reference has no CPU path: its unmodified CUDA extension (oracle/_ref) ran the full "
                                      "workload on %d B200(s), each driven by 1 host thread" % ws},
           "e2e": {"value": round(value, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if per_config:
        out["per_config"] = per_config
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C4", choices=["C1", "C2", "C4", "C5"])
    ap.add_argument("--views-per-call", type=int, default=8,
                    help="views rendered per renderer call (both arms; C4 only -- the other workloads have one view per rank)")
    ap.add_argument("--no-per-config", action="store_true", help="skip the C1/C2/C3/C5 `_C`-level timings (N = 1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (our arm; see the module doc)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of our arm only")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (B200); there is no CPU fallback")
    ws, rank, local = dist_setup(args.gpus)
    try:
        if args.impl == "reference":
            run_reference(args, ws, rank, local)
        else:
            run_ours(args, ws, rank, local)
    finally:
        if ws > 1 and dist.is_initialized():
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
