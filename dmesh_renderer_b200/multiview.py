"""Camera-sharded multi-view optimisation step (BASELINE.json north_star, SURVEY.md 8e).

The reference has no distributed code at all; views are independent, and only
three gradient tensors are summed over views (dL_dverts, dL_dvcolor,
dL_dfopacity: cuda_rasterizer/backward.cu:389-407,415 carry no batch offset).
So: the scene is replicated on every rank, rank r renders its slice of the
cameras, and ONE all-reduce(SUM) over a single packed fp32 buffer
[dL_dverts | dL_dvcolor | dL_dfopacity] = (6P + F) floats exchanges everything
that has to be exchanged.  Per-view gradients (verts_depth, faces_intense rows)
stay rank-local.  One process per GPU, torch.distributed (NCCL over NVLink 5 /
NVSwitch on the B200 box, gloo in the CPU tests); nothing else communicates.

The tet renderer takes part through tet_multiview_step.  Without vertex-position
gradients it has no dL_dverts, so PackedSceneGrads(None, verts_color,
faces_opacity) packs just [dL_dvcolor | dL_dfopacity] = (3P + F) floats.  Each
call passes the job index of its first view (first_view), so jittered rays
(ray_random_seed > 0) do not depend on how the views are sharded or split.
"""
import contextlib
from typing import Callable, Optional, Sequence, Tuple

import torch
import torch.distributed as dist


def bind_to_gpu_cpus(device_index: int, min_cores: int = 2):
    """Restrict this process (the calling thread and every thread it creates afterwards) to the CPU cores NVML lists
    as local to GPU `device_index` -- same NUMA node / PCIe root complex -- so that the pinned staging buffers
    allocated afterwards live in that node's memory and the H2D copies of several ranks do not all cross the
    socket interconnect.  Call it right after torch.cuda.set_device(local_rank), before allocating pinned memory.
    Returns the core list, or None when NVML is unavailable or fewer than `min_cores` of those cores are usable
    (e.g. a container cpuset on the other socket): then nothing is changed."""
    import os
    try:
        import pynvml
        pynvml.nvmlInit()
        uuid = getattr(torch.cuda.get_device_properties(device_index), "uuid", None)
        if uuid is not None:
            handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(uuid)).encode())
        else:
            handle = pynvml.nvmlDeviceGetHandleByIndex(device_index)
        words = ((os.cpu_count() or 64) + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(handle, words)
        cores = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
        local = sorted(cores & os.sched_getaffinity(0))
        if len(local) < min_cores:
            return None
        os.sched_setaffinity(0, local)
        return local
    except Exception:
        return None


def shard_views(num_views: int, rank: int, world_size: int) -> range:
    """Contiguous slice of the cameras owned by `rank` (SURVEY 8e: rank r renders
    views r*B/G .. (r+1)*B/G - 1; remainders go to the first ranks)."""
    base, rem = divmod(num_views, world_size)
    start = rank * base + min(rank, rem)
    return range(start, start + base + (1 if rank < rem else 0))


class PackedSceneGrads:
    """Scene leaves (verts, verts_color, faces_opacity) whose .grad tensors are
    views into ONE contiguous fp32 buffer, so the step needs a single collective.
    Layout [verts | verts_color | faces_opacity], 6P + F floats.  verts=None gives
    the tet renderer's layout without positions, [verts_color | faces_opacity],
    3P + F floats; `leaves` then holds the two tensors, and only TetRenderer calls
    can use it as a sink (see direct()).

    bg (optional): the background colour, a float32 tensor of 3 elements that the
    renderers' settings carry.  Its gradient slot is appended after faces_opacity
    (and before any padding), so the one all-reduce sums it too and the ranks'
    backgrounds stay equal; the renderers' backward passes reach it through
    ordinary autograd accumulation into the bound .grad view.  `leaves` does not
    include it.

    On a CUDA job with world_size > 1 the buffer is allocated in SYMMETRIC memory
    (torch.distributed._symmetric_memory: peer-mapped on every rank + an NVLS multicast
    address) and the all-reduce is the hand-written in-switch reduction kernel of
    csrc/collective.cu (multimem.ld_reduce / multimem.st); without multicast support
    (or on CPU / gloo) it is torch.distributed.all_reduce.  Construct it collectively:
    every rank of `group` must create its PackedSceneGrads at the same point."""

    def __init__(self, verts: torch.Tensor, verts_color: torch.Tensor, faces_opacity: torch.Tensor, group=None,
                 use_nvls: Optional[bool] = None, bg: Optional[torch.Tensor] = None):
        self.leaves = [t for t in (verts, verts_color, faces_opacity) if t is not None]
        if len(self.leaves) < 2 or verts_color is None or faces_opacity is None:
            raise ValueError("PackedSceneGrads needs verts_color and faces_opacity")
        if bg is not None and (bg.dtype != torch.float32 or bg.numel() != 3 or not bg.is_leaf):
            raise ValueError("PackedSceneGrads: bg must be a float32 leaf tensor of 3 elements")
        self.bg = bg
        self.group = group
        device = verts_color.device
        n = sum(t.numel() for t in self._slots())
        self._nvls = None
        # which collective all_reduce() runs and, for the fallback, why: "nvls" | "nccl: <reason>" | "none: <reason>"
        self.collective = "nccl: use_nvls=False" if use_nvls is False else "none: single process"
        full = None
        if use_nvls is not False:
            full = self._try_symmetric(n, device, group)
        if full is None:
            full = torch.zeros(n, dtype=torch.float32, device=device)
        self._full = full              # padded to a multiple of 4 * world_size floats in the NVLS case
        self.flat = full[:n]
        for t in self._slots():
            if not t.requires_grad:
                t.requires_grad_(True)
        self.bind()

    def _slots(self):
        return self.leaves + ([self.bg] if self.bg is not None else [])

    def bind(self):
        """(Re-)attach the leaves' .grad tensors to the packed buffer.  Anything that REPLACES .grad --
        optimizer.zero_grad() with its default set_to_none=True, `leaf.grad = None` -- silently disconnects a leaf:
        autograd would then accumulate into a fresh tensor and all_reduce() would exchange a stale buffer.  zero_(),
        direct() and all_reduce() therefore call this first; a gradient found in a foreign tensor is moved into the
        packed buffer so that nothing is lost.  Returns the number of leaves (bg included) that had to be re-attached."""
        o, fixed = 0, 0
        for t in self._slots():
            view = self.flat[o:o + t.numel()].view_as(t)
            g = t.grad
            if g is None or g.data_ptr() != view.data_ptr() or g.shape != view.shape or g.dtype != view.dtype:
                if g is not None:
                    view.copy_(g)
                t.grad = view
                fixed += 1
            o += t.numel()
        return fixed

    def _try_symmetric(self, n, device, group):
        if not (device.type == "cuda" and dist.is_available() and dist.is_initialized()):
            self.collective = "none: single process" if not (dist.is_available() and dist.is_initialized()) \
                else "%s: tensors on %s" % (dist.get_backend(group), device.type)
            return None
        ws = dist.get_world_size(group)
        if ws <= 1 or dist.get_backend(group) != "nccl":
            self.collective = "none: world size 1" if ws <= 1 else "%s: not an NCCL group" % dist.get_backend(group)
            return None
        ok, full, hdl, why = 1, None, None, ""
        try:
            import torch.distributed._symmetric_memory as symm_mem
            pg = group if group is not None else dist.group.WORLD
            if hasattr(symm_mem, "enable_symm_mem_for_group"):
                import warnings
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    symm_mem.enable_symm_mem_for_group(pg.group_name)
            n_pad = -(-n // (4 * ws)) * (4 * ws)
            full = symm_mem.empty(n_pad, dtype=torch.float32, device=device)
            full.zero_()
            hdl = symm_mem.rendezvous(full, pg)
            if not hdl.multicast_ptr:     # no NVLS multicast object behind the allocation (no NVSwitch / disabled)
                ok, why = 0, "symmetric allocation has no multicast address (no NVSwitch multicast on this node)"
            # flag words for the in-kernel cross-GPU barriers (symmetric, zeroed) + this GPU's control words
            flags = symm_mem.empty(256, dtype=torch.int32, device=device)
            flags.zero_()
            fh = symm_mem.rendezvous(flags, pg)
            ctl = torch.zeros(4, dtype=torch.int32, device=device)
        except Exception as ex:           # symmetric memory unavailable in this build / on this node
            ok, why = 0, "symmetric memory setup failed: %s: %s" % (type(ex).__name__, str(ex).splitlines()[0][:200] if str(ex) else "")
        # all ranks must take the same path
        flag = torch.tensor([ok], dtype=torch.int32, device=device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
        if int(flag.item()) != 1:
            self.collective = "nccl: " + (why or "another rank could not set up symmetric memory")
            return None
        torch.cuda.synchronize(device)
        dist.barrier(group)            # every rank's flag words are zero before anybody signals
        self._nvls = (hdl, int(hdl.multicast_ptr) + int(getattr(hdl, "offset", 0) or 0), full.numel(), dist.get_rank(group), ws)
        self._flags = (flags, fh, int(fh.buffer_ptrs_dev), ctl)
        self._epoch = 0
        self.collective = "nvls"
        return full

    def zero_(self):
        self._full.zero_()
        self.bind()

    @contextlib.contextmanager
    def direct(self):
        """While active, TriRenderer and TetRenderer calls on these leaves accumulate their scene gradients straight
        into the packed buffer from the backward kernels (no intermediate gradient tensors, no autograd accumulation
        kernels).  The leaves must be passed to the renderer themselves (not views or functions of them); gradient
        hooks on them do not see this contribution.  The choice is made at forward time, so backward may run later.
        A tet call adds into the verts slot only when its vertex-position gradients run; a buffer without that slot
        (verts=None) serves tet calls only.  Camera, intensity and other per-view gradients always go through
        autograd."""
        from . import _C
        self.bind()
        _C._grad_sinks.append(self)
        try:
            yield self
        finally:
            _C._grad_sinks.remove(self)

    def all_reduce(self, group=None, async_op=False):
        self.bind()
        if self._nvls is not None:
            import ctypes
            from . import _lib
            _, mc, n_pad, rank, ws = self._nvls
            stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            # one launch: barrier ("every rank's gradients are complete") -> in-switch reduce + broadcast of this
            # rank's slice -> barrier ("every slice has been broadcast"), all inside the kernel
            self._epoch += 1
            flags, fh, peer_ptrs, ctl = self._flags
            _lib.check(_lib.load().dmr_nvls_allreduce_sum_f32_fused(ctypes.c_void_p(mc), n_pad, rank, ws,
                                                                    ctypes.c_void_p(peer_ptrs), ctypes.c_void_p(ctl.data_ptr()),
                                                                    self._epoch, stream))
            return None
        group = group if group is not None else self.group
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
            return dist.all_reduce(self.flat, op=dist.ReduceOp.SUM, group=group, async_op=async_op)
        return None


def multiview_step(render: Callable, scene_grads: PackedSceneGrads, faces: torch.Tensor, mv_mats: torch.Tensor,
                   proj_mats: torch.Tensor, verts_depth: torch.Tensor, faces_intense: torch.Tensor,
                   cotangent_fn: Callable[[torch.Tensor, torch.Tensor], Tuple[torch.Tensor, torch.Tensor]],
                   group=None, views_per_call: Optional[int] = None) -> Sequence[torch.Tensor]:
    """One optimisation step on this rank's cameras.

    render            a TriRenderer-like callable (verts, faces, verts_color, faces_opacity,
                      mv, proj, verts_depth, faces_intense) -> (color, depth)
    mv_mats ...       THIS RANK's slice: [B_local,4,4], [B_local,P], [B_local,F]
    cotangent_fn      (color, depth) -> (dL_dcolor, dL_ddepth)   (e.g. gradient of an image loss); when the
                      renderer also returns an alpha image (TriRenderer(..., return_alpha=True)):
                      (color, depth, alpha) -> (dL_dcolor, dL_ddepth, dL_dalpha)
    views_per_call    split the local views into calls of this many views (None = one call)

    After the call every rank holds the view-summed gradients of the whole job in
    scene_grads.leaves[i].grad (and scene_grads.bg.grad).  Returns the list of (color, depth[, alpha]) outputs.
    """
    verts, verts_color, faces_opacity = scene_grads.leaves
    scene_grads.zero_()
    B = mv_mats.shape[0]
    step = views_per_call or max(B, 1)
    outs = []
    with scene_grads.direct():
        for s in range(0, B, step):
            e = min(B, s + step)
            images = render(verts, faces, verts_color, faces_opacity, mv_mats[s:e], proj_mats[s:e],
                            verts_depth[s:e], faces_intense[s:e])        # (color, depth) or (color, depth, alpha)
            torch.autograd.backward(list(images), list(cotangent_fn(*images)))
            outs.append(tuple(x.detach() for x in images))
    scene_grads.all_reduce(group)
    return outs


def tet_multiview_step(render: Callable, scene_grads: PackedSceneGrads, verts: torch.Tensor, faces: torch.Tensor,
                       tets: torch.Tensor, face_tets: torch.Tensor, tet_faces: torch.Tensor, mv_mats: torch.Tensor,
                       proj_mats: torch.Tensor, verts_depth: torch.Tensor, faces_intense: torch.Tensor,
                       cotangent_fn: Callable[[torch.Tensor, torch.Tensor], Tuple[torch.Tensor, torch.Tensor]],
                       group=None, views_per_call: Optional[int] = None,
                       first_view: int = 0) -> Sequence[Tuple[torch.Tensor, torch.Tensor, torch.Tensor]]:
    """One optimisation step of the tet renderer on this rank's cameras (multiview_step for TetRenderer).

    render            a TetRenderer-like callable (verts, faces, verts_color, faces_opacity, mv, proj, verts_depth,
                      faces_intense, tets, face_tets, tet_faces, first_view=...) -> (color, depth, active)
    scene_grads       PackedSceneGrads(verts, verts_color, faces_opacity) (6P + F floats; verts gets gradients when the
                      renderer's vertex_grads is on) or PackedSceneGrads(None, verts_color, faces_opacity) (3P + F)
    verts             the scene's vertex positions; when scene_grads has a verts slot, its own verts leaf
    mv_mats ...       THIS RANK's slice: [B_local,4,4], [B_local,P], [B_local,F]
    cotangent_fn      (color, depth) -> (dL_dcolor, dL_ddepth); when the renderer also returns an alpha image
                      (TetRenderer(..., return_alpha=True)): (color, depth, alpha) -> (dL_dcolor, dL_ddepth, dL_dalpha)
    views_per_call    split the local views into calls of this many views (None = one call)
    first_view        index of mv_mats[0] among all the job's cameras: shard_views(B, rank, world_size).start.  Call s
                      renders with first_view + s, so jittered rays match one call over all views.

    After the call every rank holds the view-summed gradients of the whole job in the leaves' .grad (and
    scene_grads.bg.grad).  Returns the list of (color, depth, active[, alpha]) outputs.
    """
    if len(scene_grads.leaves) == 3 and verts is not scene_grads.leaves[0]:
        raise ValueError("tet_multiview_step: scene_grads holds vertex positions, so verts must be its verts leaf "
                         "(scene_grads.leaves[0])")
    verts_color, faces_opacity = scene_grads.leaves[-2:]
    scene_grads.zero_()
    B = mv_mats.shape[0]
    step = views_per_call or max(B, 1)
    outs = []
    with scene_grads.direct():
        for s in range(0, B, step):
            e = min(B, s + step)
            out = render(verts, faces, verts_color, faces_opacity, mv_mats[s:e], proj_mats[s:e], verts_depth[s:e],
                         faces_intense[s:e], tets, face_tets, tet_faces, first_view=first_view + s)
            images = out[:2] + out[3:]                           # (color, depth) or (color, depth, alpha)
            torch.autograd.backward(list(images), list(cotangent_fn(*images)))
            outs.append((out[0].detach(), out[1].detach(), out[2]) + tuple(x.detach() for x in out[3:]))
    scene_grads.all_reduce(group)
    return outs
