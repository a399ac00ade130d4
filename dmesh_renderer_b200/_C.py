"""`_C` shim: the four entry points of the reference's pybind module
(/root/reference/ext.cpp:4-12, render.h:10-111) with the same names, positional
signatures, return tuples, validation messages and edge-case behaviour
(render.cu:29-412), implemented on top of the C ABI of libdmesh_b200.so.

PyTorch is used only for device memory (output / state tensors are allocated
through the caching allocator exactly like the reference's torch::full /
resize_ lambdas, render.cu:18-24,87-100) and for the current stream.  All
compute happens in the hand-written sm_100a kernels behind the C ABI; there is
no fallback.
"""
import ctypes

import torch

from . import _lib

NUM_CHANNELS = 3  # cuda_rasterizer/config.h:4


def _err(msg):
    # AT_ERROR -> c10::Error -> RuntimeError on the Python side
    raise RuntimeError(msg)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None and t.numel() > 0 else ctypes.c_void_p(0)


def _f32(t, name):
    if t.dtype != torch.float32:
        # the reference's .data<float>() throws for any other dtype
        raise RuntimeError("expected scalar type Float but found %s for %s" % (str(t.dtype).replace("torch.", ""), name))
    return t.contiguous()


def _i32(t, name):
    if t.dtype != torch.int32:
        raise RuntimeError("expected scalar type Int but found %s for %s" % (str(t.dtype).replace("torch.", ""), name))
    return t.contiguous()


def _require_cuda(*ts):
    for t in ts:
        if not t.is_cuda:
            raise RuntimeError("dmesh_renderer_b200 is CUDA-only (sm_100a); got a %s tensor. There is no CPU fallback." % t.device)


class _Pinned:
    """Pinned int32 words for the num_rendered read-back (the single host<->device synchronisation of a forward
    call, as in rasterizer_impl.cu:287-292).  Every forward call in flight owns ITS OWN word, taken from a small
    per-device pool and given back when the call has read it: the split API (tri_forward_begin / _finish) allows
    several calls between their two phases, and ctypes releases the GIL inside dmr_wait_i32, so two Python threads
    can render on one GPU at the same time -- neither may see the other's count.  list.pop / list.append are
    atomic under the GIL."""
    _free = {}

    @classmethod
    def acquire(cls, device, n=1):
        key = (device.index if device.index is not None else torch.cuda.current_device(), n)
        pool = cls._free.setdefault(key, [])
        try:
            return pool.pop()
        except IndexError:
            t = torch.zeros(n, dtype=torch.int32).pin_memory()
            return (t, t.numpy(), ctypes.c_void_p(t.data_ptr()), key)   # tensor, numpy view (cheap host reads), pointer, pool

    @classmethod
    def release(cls, slot):
        if slot is not None:
            cls._free[slot[3]].append(slot)


def _stream():
    # raw handle of the current stream of the current device; torch.cuda.current_stream() costs ~10 us of Python
    # per call (device-index resolution, Stream object), and a forward+backward needs it four times
    return ctypes.c_void_p(torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice()))


class _on_device:
    """`with torch.cuda.device(dev)` without its cost when `dev` already is the current device (the normal case:
    one process per GPU, torch.cuda.set_device(rank))."""
    __slots__ = ("ctx",)

    def __init__(self, dev):
        idx = dev.index
        self.ctx = None if idx is None or idx == torch._C._cuda_getDevice() else torch.cuda.device(dev)

    def __enter__(self):
        if self.ctx is not None:
            self.ctx.__enter__()

    def __exit__(self, *exc):
        if self.ctx is not None:
            return self.ctx.__exit__(*exc)
        return False


_SENTINEL = -2 ** 31          # num_rendered is never negative
_last_R = {}                  # (renderer, B, P, F, T, W, H) -> num_rendered of the previous call


def _arm(pinned):
    pinned[1][0] = _SENTINEL


def _speculative_binning(lib, key, u8):
    """Binning buffer sized from the previous call with the same shapes (+25%), allocated while the GPU is still
    busy with phase 1.  Returns (buffer, capacity in instances) or (None, 0) on the first call."""
    prev = _last_R.get(key)
    if not prev:
        return None, 0
    cap = min(prev + prev // 4 + 1024, _MAX_R)
    return torch.empty(lib.dmr_binning_bytes(cap), **u8), cap


_MAX_R = (1 << 30) - 1          # the sort's descriptors carry 30-bit prefixes (csrc/radix_sort.cu)


def _wait_R(lib, pinned, key, spec, u8):
    """The one host<->device synchronisation of a forward call (rasterizer_impl.cu:287-292): wait for
    num_rendered, return (R, binning buffer)."""
    _lib.check(lib.dmr_wait_i32(pinned[2], _SENTINEL, _stream()))
    R = int(pinned[1][0])
    if R < 0 or R > _MAX_R:         # the scan saturates at 2^32 - 1, which arrives here as a negative int32
        raise RuntimeError("dmesh_renderer_b200: %s tile instances exceed the supported maximum of 2^30 - 1 "
                           "(the reference's int limit is 2^31 - 1); render fewer views per call" %
                           ("more than 2^31" if R < 0 else str(R)))
    _last_R[key] = R
    need = lib.dmr_binning_bytes(R) if R > 0 else 0
    if spec is not None and spec.numel() >= need:
        return R, spec
    return R, torch.empty(need, **u8)


def _read_R(lib, pinned, key):
    """Wait for num_rendered (see _wait_R) without touching buffers."""
    _lib.check(lib.dmr_wait_i32(pinned[2], _SENTINEL, _stream()))
    R = int(pinned[1][0])
    if R < 0 or R > _MAX_R:
        raise RuntimeError("dmesh_renderer_b200: %s tile instances exceed the supported maximum of 2^30 - 1 "
                           "(the reference's int limit is 2^31 - 1); render fewer views per call" %
                           ("more than 2^31" if R < 0 else str(R)))
    _last_R[key] = R
    return R


class _Inverses:
    """inverse(mv), inverse(proj) with the bits torch.inverse produces (reference dmesh_renderer/__init__.py:62-63,
    298-299) from ONE kernel launch (csrc/inverse.cu: the same LU / triangular-solve arithmetic, one thread per
    matrix) instead of ~24 library kernels and the two device synchronisations torch.inverse performs to look at
    LAPACK's `info` vector.  The kernel writes `info` straight into pinned host memory; it is examined after the
    synchronisation the forward call needs anyway (num_rendered), and a singular matrix raises the same error,
    through torch.inverse itself.  `mv` / `proj` are contiguous copies of the inputs written by the same kernel
    (the API passes transposed views).  Anything but fp32 CUDA [B,4,4] stacks takes torch.linalg.inv_ex."""
    __slots__ = ("inv_mv", "inv_proj", "mv", "proj", "mats", "host_np", "slot")
    _pinned = {}

    def __init__(self, mv_mats, proj_mats):
        self.mats = (mv_mats, proj_mats)
        self.mv, self.proj = mv_mats, proj_mats
        self.host_np = None
        self.slot = None
        native = (mv_mats.is_cuda and proj_mats.is_cuda and mv_mats.device == proj_mats.device and
                  mv_mats.dtype == torch.float32 and proj_mats.dtype == torch.float32 and mv_mats.dim() == 3 and
                  mv_mats.shape == proj_mats.shape and tuple(mv_mats.shape[1:]) == (4, 4) and mv_mats.size(0) > 0)
        if native:
            dev, B = mv_mats.device, mv_mats.size(0)
            slot = self.slot = _Pinned.acquire(dev, 2 * B)      # this call's own `info` words (see _Pinned)
            with _on_device(dev):
                out = torch.empty((4, B, 4, 4), dtype=torch.float32, device=dev)
                _lib.check(_lib.load().dmr_camera_inverses(B, _ptr(mv_mats), *mv_mats.stride(), _ptr(proj_mats),
                                                           *proj_mats.stride(), _ptr(out), slot[2], _stream()))
            self.mv, self.proj, self.inv_mv, self.inv_proj = out[0], out[1], out[2], out[3]
            self.host_np = slot[1]
            return
        self.inv_mv, info_mv = torch.linalg.inv_ex(mv_mats)
        self.inv_proj, info_pj = torch.linalg.inv_ex(proj_mats)
        info = torch.cat([info_mv.reshape(-1), info_pj.reshape(-1)])
        if mv_mats.is_cuda:
            n = info.numel()
            key = (mv_mats.device.index, -n)
            host = _Inverses._pinned.get(key)
            if host is None:
                host = _Inverses._pinned[key] = torch.zeros(max(n, 1), dtype=torch.int32).pin_memory()
            if n:
                host[:n].copy_(info, non_blocking=True)
            self.host_np = host[:n].numpy()
        else:
            self.check(info)

    def check(self, *infos):
        """Call after the current stream has been synchronised."""
        if infos:
            bad = any(bool(i.any()) for i in infos)
        else:
            bad = self.host_np is not None and bool(self.host_np.any())
        if self.slot is not None:
            _Pinned.release(self.slot)
            self.slot = self.host_np = None
        if bad:
            torch.inverse(self.mats[0])   # raises torch's own "singular matrix" error
            torch.inverse(self.mats[1])


def _check_common(verts, faces, mv_mats, proj_mats, inv_mv_mats, inv_proj_mats, verts_depth, faces_intense, tri):
    # messages follow render.cu:49-79 (tri) and 237-267 (tet)
    if verts.dim() != 2 or verts.size(1) != 3:
        _err("verts must have dimensions (num_points, 3)")
    if faces.dim() != 2 or faces.size(1) != 3:
        _err("faces must have dimensions (num_faces, 3)")
    names = ("(B, 4, 4)" if tri else "(batch_size, 4, 4)")
    for t, n in ((mv_mats, "mv_mats"), (proj_mats, "proj_mats"), (inv_mv_mats, "inv_mv_mats"), (inv_proj_mats, "inv_proj_mats")):
        if t.dim() != 3 or t.size(1) != 4 or t.size(2) != 4:
            _err("%s must have dimensions %s" % (n, names))
    if verts_depth.dim() != 2 or verts_depth.size(1) != verts.size(0):
        _err("verts_depth must have dimensions (B, num_points,)" if tri else "verts_depth must have dimensions (batch_size, num_verts)")
    if faces_intense.dim() != 2 or faces_intense.size(1) != faces.size(0):
        _err("faces_intense must have dimensions (B, num_faces,)" if tri else "faces_intense must have dimensions (batch_size, num_faces)")


# ---------------------------------------------------------------------------
# tri renderer
# ---------------------------------------------------------------------------
class _TriPending:
    """Forward call between phase 1 (enqueued) and phase 2 (needs R and the inverse matrices)."""
    __slots__ = ("dims", "dev", "bg", "bufs", "outs", "pinned", "empty")


def tri_forward_begin(background, verts, faces, verts_color, faces_opacity, mv_mats, proj_mats, verts_depth,
                      faces_intense, image_height, image_width):
    """Validate, allocate state, enqueue phase 1 (preprocess + records + scan) on the current stream.
    Split out of render_tris so that a caller can do host work (allocate the speculative binning buffer, prepare the
    phase-2 arguments) while the GPU runs phase 1.  Returns a pending-call object for tri_forward_finish."""
    if verts.dim() != 2 or verts.size(1) != 3:
        _err("verts must have dimensions (num_points, 3)")
    if faces.dim() != 2 or faces.size(1) != 3:
        _err("faces must have dimensions (num_faces, 3)")
    if verts_color.dim() != 2 or verts_color.size(0) != verts.size(0):
        _err("vert color must have dimensions (num_points, N)")
    if faces_opacity.dim() != 1 or faces_opacity.size(0) != faces.size(0):
        _err("face opacity must have dimensions (num_faces,)")
    for t, n in ((mv_mats, "mv_mats"), (proj_mats, "proj_mats")):
        if t.dim() != 3 or t.size(1) != 4 or t.size(2) != 4:
            _err("%s must have dimensions (B, 4, 4)" % n)
    # verts_depth=None (an extension of the reference API): the renderer uses the NDC z it computes itself
    if verts_depth is not None and (verts_depth.dim() != 2 or verts_depth.size(1) != verts.size(0)):
        _err("verts_depth must have dimensions (B, num_points,)")
    if faces_intense.dim() != 2 or faces_intense.size(1) != faces.size(0):
        _err("faces_intense must have dimensions (B, num_faces,)")
    _require_cuda(background, verts, faces, verts_color, faces_opacity, mv_mats, proj_mats, faces_intense)
    if verts_depth is not None:
        _require_cuda(verts_depth)
    lib = _lib.load()
    B, P, F = mv_mats.size(0), verts.size(0), faces.size(0)
    H, W = int(image_height), int(image_width)
    dev = verts.device
    if verts_color.size(1) != NUM_CHANNELS:
        _err("vert color must have dimensions (num_points, 3)")
    st = _TriPending()
    st.dims, st.dev, st.empty = (B, P, F, W, H), dev, P == 0
    if st.empty:
        return st
    with _on_device(dev):
        u8 = dict(dtype=torch.uint8, device=dev)
        st.bg = _f32(background, "background")
        verts_c, faces_c = _f32(verts, "verts"), _i32(faces, "faces")
        vcol, fopa = _f32(verts_color, "verts_color"), _f32(faces_opacity, "faces_opacity")
        mv, pj = _f32(mv_mats, "mv_mats"), _f32(proj_mats, "proj_mats")
        vdep = _f32(verts_depth, "verts_depth") if verts_depth is not None else None
        fint = _f32(faces_intense, "faces_intense")
        sizes = (ctypes.c_size_t * 3)()
        _lib.check(lib.dmr_tri_state_bytes(B, P, F, W, H, sizes))
        st.bufs = [torch.empty(sizes[0], **u8), torch.empty(sizes[1], **u8), torch.empty(sizes[2], **u8)]
        st.outs = [torch.empty((B, NUM_CHANNELS, H, W), dtype=torch.float32, device=dev),
                   torch.empty((B, 1, H, W), dtype=torch.float32, device=dev)]
        st.pinned = _Pinned.acquire(dev)     # released by tri_forward_finish
        _arm(st.pinned)
        _lib.check(lib.dmr_tri_forward_bin(B, P, F, W, H, _ptr(verts_c), _ptr(faces_c), _ptr(vcol), _ptr(fopa), _ptr(mv),
                                           _ptr(pj), _ptr(vdep), _ptr(fint), _ptr(st.bufs[0]), _ptr(st.bufs[1]),
                                           st.pinned[2], _stream()))
    return st


def tri_forward_finish(st, inv_mv_mats, inv_proj_mats, inverses=None, speculative=False):
    """Phase 2 of a forward call started by tri_forward_begin: the one host sync (R), binning buffer, sort, render.
    `inverses`: the _Inverses object the matrices came from, whose deferred singularity check runs after the sync.
    `speculative`: launch phase 2 BEFORE num_rendered has reached the host, on a binning buffer sized from the
    previous call with the same shapes (+25 %): the phase-2 kernels read the instance count on the device, so the GPU
    goes straight from the scan into the binning kernels while the host is still waiting for the 4-byte read-back
    (the reference drains the pipeline there, rasterizer_impl.cu:287-299).  If the scene grew past the buffer, the
    kernels emit nothing and phase 2 is simply run again with an exact buffer.  In this mode element 0 of the result is
    the CAPACITY the binning buffer was laid out for (>= num_rendered); pass it to render_tris_backward as `R`."""
    for t, n in ((inv_mv_mats, "inv_mv_mats"), (inv_proj_mats, "inv_proj_mats")):
        if t.dim() != 3 or t.size(1) != 4 or t.size(2) != 4:
            _err("%s must have dimensions (B, 4, 4)" % n)
    B, P, F, W, H = st.dims
    dev = st.dev
    lib = _lib.load()
    with _on_device(dev):
        u8 = dict(dtype=torch.uint8, device=dev)
        if st.empty:
            # render.cu:88-89,105: zero images (not background), empty state
            z = torch.zeros
            if inverses is not None:
                torch.cuda.current_stream().synchronize()
                inverses.check()
            return (0, z((B, NUM_CHANNELS, H, W), dtype=torch.float32, device=dev),
                    z((B, 1, H, W), dtype=torch.float32, device=dev),
                    torch.empty(0, **u8), torch.empty(0, **u8), torch.empty(0, **u8), torch.empty(0, **u8))
        _require_cuda(inv_mv_mats, inv_proj_mats)
        imv, ipj = _f32(inv_mv_mats, "inv_mv_mats"), _f32(inv_proj_mats, "inv_proj_mats")
        key = ("tri", B, P, F, 0, W, H)
        spec, cap = _speculative_binning(lib, key, u8)
        point_buf, face_buf, img_buf = st.bufs
        out_color, out_depth = st.outs
        # everything that does not depend on R is prepared before the wait
        a = (_ptr(st.bg), _ptr(imv), _ptr(ipj), _ptr(point_buf), _ptr(face_buf))
        b2 = (_ptr(img_buf), _ptr(out_color), _ptr(out_depth), _stream())
        try:
            if speculative and spec is not None:
                # phase 2 goes out first; the wait below overlaps with it
                _lib.check(lib.dmr_tri_forward_render(B, P, F, W, H, cap, *a, _ptr(spec), *b2))
                R = _read_R(lib, st.pinned, key)
                bin_buf = spec
                if R > cap:     # the scene outgrew the speculative buffer: nothing was emitted, run phase 2 again
                    cap = R
                    bin_buf = torch.empty(lib.dmr_binning_bytes(cap), **u8)
                    _lib.check(lib.dmr_tri_forward_render(B, P, F, W, H, cap, *a, _ptr(bin_buf), *b2))
                R = cap         # the layout count of the binning buffer (see the docstring)
            else:
                # (Measured and rejected: one native call that waits for R and launches phase 2 without returning to
                # Python in between -- 1163 vs 1159 views/s at C2: the bubble is the D2H + launch latency, not the
                # interpreter.)
                R, bin_buf = _wait_R(lib, st.pinned, key, spec, u8)   # the one sync: R sizes the binning buffer
                _lib.check(lib.dmr_tri_forward_render(B, P, F, W, H, R, *a, _ptr(bin_buf), *b2))
        finally:
            _Pinned.release(st.pinned)
            st.pinned = None
        if inverses is not None:
            inverses.check()
    return R, out_color, out_depth, point_buf, face_buf, bin_buf, img_buf


def render_tris(background, verts, faces, verts_color, faces_opacity, mv_mats, proj_mats, inv_mv_mats, inv_proj_mats,
                verts_depth, faces_intense, image_height, image_width):
    """RasterizeTrianglesCUDA (render.cu:29-132).
    Returns (num_rendered, color[B,3,H,W], depth[B,1,H,W], pointBuffer, faceBuffer, binningBuffer, imgBuffer)."""
    # shape errors are reported before anything is enqueued, in the reference's order (render.cu:49-79)
    if verts.dim() == 2 and verts.size(1) == 3 and faces.dim() == 2 and faces.size(1) == 3 and \
            verts_color.dim() == 2 and verts_color.size(0) == verts.size(0) and \
            faces_opacity.dim() == 1 and faces_opacity.size(0) == faces.size(0):
        _check_common(verts, faces, mv_mats, proj_mats, inv_mv_mats, inv_proj_mats, verts_depth, faces_intense, True)
    st = tri_forward_begin(background, verts, faces, verts_color, faces_opacity, mv_mats, proj_mats, verts_depth,
                           faces_intense, image_height, image_width)
    return tri_forward_finish(st, inv_mv_mats, inv_proj_mats)


# Gradient sinks (multiview.PackedSceneGrads.direct()): while one is active, a renderer call whose scene tensors ARE
# the sink's leaves lets its backward kernels accumulate straight into the leaves' .grad buffers (the C ABI
# accumulates into whatever it is given) and returns None for them, instead of filling three fresh tensors that
# autograd then adds to .grad with three more kernels.  Module-global: autograd runs backward on its own thread.
_grad_sinks = []


def grad_sink_for(verts, verts_color, faces_opacity, tet=False):
    """The innermost active sink whose leaves are exactly these tensors.  A sink without positions
    (PackedSceneGrads(None, verts_color, faces_opacity)) holds no verts slot; only a tet call (`tet=True`) may match
    it, on verts_color and faces_opacity alone."""
    for sink in reversed(_grad_sinks):
        if len(sink.leaves) == 3:
            xs = (verts, verts_color, faces_opacity)
        elif tet:
            xs = (verts_color, faces_opacity)
        else:
            continue
        ok = True
        for x, leaf in zip(xs, sink.leaves):
            g = leaf.grad
            if not (x is leaf or (x.data_ptr() == leaf.data_ptr() and x.shape == leaf.shape and x.dtype == leaf.dtype)) \
                    or g is None or g.dtype != torch.float32 or not g.is_contiguous() or g.shape != leaf.shape \
                    or g.device != x.device or not leaf.is_leaf:
                ok = False
                break
        if ok:
            return sink
    return None


def render_tris_backward(background, verts, faces, verts_color, faces_opacity, mv_mats, proj_mats, inv_mv_mats,
                         inv_proj_mats, verts_depth, faces_intense, dL_dout_color, dL_dout_depth, R, pointBuffer,
                         faceBuffer, binningBuffer, imageBuffer, accumulate_into=None, deterministic=False,
                         camera_grads=False, exact_vertex_grads=False, dL_dout_alpha=None, background_grad=False):
    """RasterizeTrianglesBackwardCUDA (render.cu:134-208).
    Returns (dL_dverts[P,3], dL_dvcolor[P,3], dL_dfopacity[F], dL_dvdepth[B,P], dL_dfintense[B,F]).
    `accumulate_into` (beyond the reference's 18 arguments): existing contiguous fp32 (dL_dverts, dL_dvcolor,
    dL_dfopacity) tensors that the gradients are ADDED to (and that are returned) instead of fresh zero tensors.
    `deterministic`: run-to-run reproducible gradients (64-bit fixed-point accumulation, dmr_tri_backward_deterministic).
    `camera_grads`: also return dL_dmv_mats, dL_dproj_mats [B,4,4] (gradients with respect to the mv_mats / proj_mats
    tensors passed here, through the rays; dmr_tri_backward_camera) as two more elements.
    `exact_vertex_grads`: dL_dverts is the exact derivative of the rendered image instead of the reference's formula
    (which differentiates t in place of the second barycentric v); the other gradients are unchanged
    (dmr_tri_backward_exact).
    `dL_dout_alpha`: cotangent [B,1,H,W] of the alpha image (tri_alpha); it changes dL_dfopacity only
    (dmr_tri_backward_alpha, in every mode above).
    `background_grad`: also return dL_dbackground, float32 [3], as the last element (dmr_tri_background_grad; zero
    when P == 0, where the images do not depend on the background)."""
    lib = _lib.load()
    B, P, F = mv_mats.size(0), verts.size(0), faces.size(0)
    H, W = dL_dout_color.size(2), dL_dout_color.size(3)
    dev = verts.device
    with _on_device(dev):
        # the five zero-initialised gradient tensors of render.cu:166-171, carved out of ONE allocation
        # (one memset instead of five); each starts on a 16-byte boundary
        sizes = [3 * P, NUM_CHANNELS * P, F, B * P, B * F] + ([16 * B, 16 * B] if camera_grads else [])
        if accumulate_into is not None:
            sizes[0] = sizes[1] = sizes[2] = 0
        offs, o = [], 0
        for n in sizes:
            offs.append(o)
            o += (n + 3) // 4 * 4
        flat = torch.zeros(max(o, 1), dtype=torch.float32, device=dev)
        if F != 0 and P != 0 and R > 0:
            _require_cuda(dL_dout_color, dL_dout_depth)
            bg = _f32(background, "background")
            imv, ipj = _f32(inv_mv_mats, "inv_mv_mats"), _f32(inv_proj_mats, "inv_proj_mats")
            gc, gd = _f32(dL_dout_color, "dL_dout_color"), _f32(dL_dout_depth, "dL_dout_depth")
            base = flat.data_ptr()   # the kernels are enqueued before the five views below are even created
            gp = [ctypes.c_void_p(base + 4 * off) for off in offs]
            if accumulate_into is not None:
                gp[:3] = [ctypes.c_void_p(t.data_ptr()) for t in accumulate_into]
            a = (B, P, F, W, H, int(R), _ptr(bg), _ptr(imv), _ptr(ipj), _ptr(pointBuffer), _ptr(faceBuffer),
                 _ptr(binningBuffer), _ptr(imageBuffer), _ptr(gc), _ptr(gd), gp[0], gp[1], gp[2], gp[3], gp[4])
            # scratch of the call (statistics per (view, face), per-vertex accumulators): the state buffers saved for
            # backward are only read.  The caching allocator reuses the block for later work on the same stream.
            if dL_dout_alpha is not None:
                # the workspace of the mode it modifies
                det = int(bool(deterministic))
                ga = _f32(dL_dout_alpha, "dL_dout_alpha")
                if ga.numel() != B * H * W:
                    _err("dL_dout_alpha must have dimensions (B, 1, H, W)")
                nbytes = (lib.dmr_tri_backward_camera_bytes(B, P, F, W, H, det) if camera_grads else
                          lib.dmr_tri_backward_deterministic_bytes(B, P, F) if det else
                          lib.dmr_tri_backward_workspace_bytes(B, P, F))
                ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
                cam = (gp[5], gp[6]) if camera_grads else (ctypes.c_void_p(0), ctypes.c_void_p(0))
                _lib.check(lib.dmr_tri_backward_alpha(*a, det, int(bool(exact_vertex_grads)), *cam, _ptr(ga), _ptr(ws),
                                                      ws.numel(), _stream()))
            elif exact_vertex_grads:
                # the workspace of the mode it modifies: the record layout is the same
                det = int(bool(deterministic))
                nbytes = (lib.dmr_tri_backward_camera_bytes(B, P, F, W, H, det) if camera_grads else
                          lib.dmr_tri_backward_deterministic_bytes(B, P, F) if det else
                          lib.dmr_tri_backward_workspace_bytes(B, P, F))
                ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
                cam = (gp[5], gp[6]) if camera_grads else (ctypes.c_void_p(0), ctypes.c_void_p(0))
                _lib.check(lib.dmr_tri_backward_exact(*a, det, *cam, _ptr(ws), ws.numel(), _stream()))
            elif camera_grads:
                ws = torch.empty(lib.dmr_tri_backward_camera_bytes(B, P, F, W, H, int(bool(deterministic))),
                                 dtype=torch.uint8, device=dev)
                _lib.check(lib.dmr_tri_backward_camera(*a, int(bool(deterministic)), gp[5], gp[6], _ptr(ws), ws.numel(),
                                                       _stream()))
            elif deterministic:
                ws = torch.empty(lib.dmr_tri_backward_deterministic_bytes(B, P, F), dtype=torch.uint8, device=dev)
                _lib.check(lib.dmr_tri_backward_deterministic(*a, _ptr(ws), ws.numel(), _stream()))
            else:
                ws = torch.empty(lib.dmr_tri_backward_workspace_bytes(B, P, F), dtype=torch.uint8, device=dev)
                _lib.check(lib.dmr_tri_backward(*a, _ptr(ws), ws.numel(), _stream()))
        if accumulate_into is not None:
            dL_dverts, dL_dvcolor, dL_dfopacity = accumulate_into
        else:
            dL_dverts = flat[offs[0]:offs[0] + sizes[0]].view(P, 3)
            dL_dvcolor = flat[offs[1]:offs[1] + sizes[1]].view(P, NUM_CHANNELS)
            dL_dfopacity = flat[offs[2]:offs[2] + sizes[2]]
        dL_dvdepth = flat[offs[3]:offs[3] + sizes[3]].view(B, P)
        dL_dfintense = flat[offs[4]:offs[4] + sizes[4]].view(B, F)
        out = (dL_dverts, dL_dvcolor, dL_dfopacity, dL_dvdepth, dL_dfintense)
        if camera_grads:
            # [B,16] column-major = [B,4,4] gradients of the (column-major, i.e. transposed) matrix tensors given here
            out += (flat[offs[5]:offs[5] + sizes[5]].view(B, 4, 4), flat[offs[6]:offs[6] + sizes[6]].view(B, 4, 4))
        if background_grad:
            out += (_background_grad(lib.dmr_tri_background_grad_bytes, lib.dmr_tri_background_grad, B, W, H,
                                     imageBuffer, dL_dout_color, dev),)
    return out


def _background_grad(nbytes_fn, grad_fn, B, W, H, imageBuffer, dL_dout_color, dev):
    """dL/dbackground [3] fp32 of one renderer call (dmr_tri_background_grad / dmr_tet_background_grad); zero when
    the call kept no image state (tri with P == 0: zero images that do not depend on the background)."""
    out = torch.zeros(3, dtype=torch.float32, device=dev)
    if imageBuffer is None or imageBuffer.numel() == 0 or B * W * H == 0:
        return out
    _require_cuda(dL_dout_color)
    gc = _f32(dL_dout_color, "dL_dout_color")
    ws = torch.empty(nbytes_fn(B), dtype=torch.uint8, device=dev)
    _lib.check(grad_fn(B, W, H, _ptr(imageBuffer), _ptr(gc), _ptr(out), _ptr(ws), ws.numel(), _stream()))
    return out


def _alpha(fn, B, W, H, imageBuffer, dev):
    out = torch.zeros((B, 1, H, W), dtype=torch.float32, device=dev)
    if imageBuffer is not None and imageBuffer.numel() > 0 and out.numel() > 0:
        _lib.check(fn(B, W, H, _ptr(imageBuffer), _ptr(out), _stream()))
    return out


def tri_alpha(imageBuffer, B, H, W, device):
    """Alpha image [B,1,H,W] fp32 of a tri forward call: 1 - final_T (dmr_tri_alpha); zeros when P == 0 (the call's
    image buffer is empty).  Enqueue after the forward call's last phase 2."""
    with _on_device(device):
        return _alpha(_lib.load().dmr_tri_alpha, B, W, H, imageBuffer, device)


def tet_alpha(imageBuffer, B, H, W, device):
    """Alpha image [B,1,H,W] fp32 of a tet forward call: 1 - expf(final_log_T) on active pixels, 0 on inactive ones
    (dmr_tet_alpha)."""
    with _on_device(device):
        return _alpha(_lib.load().dmr_tet_alpha, B, W, H, imageBuffer, device)


def tri_depth_chain(verts, mv_mats, proj_mats, dL_dvdepth, dL_dverts, dL_dmv=None, dL_dproj=None):
    """Fused vertex depth (verts_depth=None): dL_dverts += sum_b dL_dvdepth[b] * d ndc_z / d verts, in place.
    With `dL_dmv` and `dL_dproj` (contiguous fp32 [B,4,4], e.g. from render_tris_backward(camera_grads=True)) the
    depth's chain into the matrices is added to them as well (dmr_tri_depth_chain_camera)."""
    lib = _lib.load()
    B, P = mv_mats.size(0), verts.size(0)
    if (dL_dmv is None) != (dL_dproj is None):
        _err("tri_depth_chain: pass both dL_dmv and dL_dproj, or neither")
    with _on_device(verts.device):
        # keep the contiguous copies alive in locals until the launch is enqueued (a temporary would be freed, and
        # its memory handed to the next .contiguous(), before the call)
        v, mv, pj = _f32(verts, "verts"), _f32(mv_mats, "mv_mats"), _f32(proj_mats, "proj_mats")
        if dL_dmv is None:
            _lib.check(lib.dmr_tri_depth_chain(B, P, _ptr(v), _ptr(mv), _ptr(pj), _ptr(dL_dvdepth), _ptr(dL_dverts),
                                               _stream()))
        else:
            for t, n in ((dL_dmv, "dL_dmv"), (dL_dproj, "dL_dproj")):
                if t.dtype != torch.float32 or not t.is_contiguous() or t.numel() != 16 * B:
                    _err("%s must be a contiguous float32 (B, 4, 4) tensor" % n)
            ws = torch.empty(lib.dmr_tri_depth_chain_camera_bytes(B, P), dtype=torch.uint8, device=verts.device)
            _lib.check(lib.dmr_tri_depth_chain_camera(B, P, _ptr(v), _ptr(mv), _ptr(pj), _ptr(dL_dvdepth), _ptr(dL_dverts),
                                                      _ptr(dL_dmv), _ptr(dL_dproj), _ptr(ws), ws.numel(), _stream()))
    return dL_dverts


# ---------------------------------------------------------------------------
# tet renderer
# ---------------------------------------------------------------------------
class _TetRecordCache:
    """The view-independent adjacency records of the tet renderer (one 128-byte TetRec per tet, csrc/tet.cuh)
    depend only on verts / faces / tets / face_tets / tet_faces.  Without vertex-position gradients none of them
    carries a gradient (reference dmesh_renderer/__init__.py:407-422), so in an optimisation loop they are the same
    tensors in every step: the records are built once and reused while the caller keeps passing the SAME tensor
    objects, unmodified (identity + torch's in-place version counter; weak references, so a freed tensor can never
    match a new one that happens to reuse its memory).  With vertex-position gradients (set_tet_vertex_grads) the
    optimiser updates `verts` in place every step; that bumps its version counter, so the records are rebuilt.
    Writing through `verts.data` bypasses the version counter and is not supported: the stale records would be
    reused.  One entry per device."""
    _entries = {}

    @classmethod
    def get(cls, lib, tensors, T, dev):
        import weakref
        key = dev.index if dev.index is not None else torch.cuda.current_device()
        e = cls._entries.get(key)
        if e is not None:
            refs, versions, buf = e
            if len(refs) == len(tensors) and all(r() is t for r, t in zip(refs, tensors)) and \
                    versions == tuple(t._version for t in tensors):
                return buf, 1
        buf = torch.empty(lib.dmr_tet_records_bytes(T), dtype=torch.uint8, device=dev)
        try:
            cls._entries[key] = ([weakref.ref(t) for t in tensors], tuple(t._version for t in tensors), buf)
        except TypeError:
            cls._entries.pop(key, None)
        return buf, 0

    @classmethod
    def clear(cls):
        cls._entries.clear()


def render_tets(background, verts, faces, verts_color, faces_opacity, mv_mats, proj_mats, inv_mv_mats, inv_proj_mats,
                verts_depth, faces_intense, tets, face_tets, tet_faces, image_height, image_width, ray_random_seed,
                inverses=None, first_view=0):
    """RenderFTetsCUDA (render.cu:213-336).
    Returns (color[B,3,H,W], depth[B,1,H,W], active_f32[B,H,W], pointBuffer, faceBuffer, binningBuffer, imgBuffer).
    `inverses` (beyond the reference's 17 arguments): see tri_forward_finish.
    `first_view` (beyond the reference's 17 arguments): index of this call's view 0 in a larger job.  With
    ray_random_seed > 0 the jitter of a view then depends only on its index in the job, not on the call that renders
    it (dmr_tet_forward_render_views); 0, the default, gives the reference's rays.
    The cached adjacency records (_TetRecordCache) travel with the returned face buffer as its attribute
    `tet_records`, for render_tets_backward."""
    if verts.dim() != 2 or verts.size(1) != 3:
        _err("verts must have dimensions (num_points, 3)")
    if faces.dim() != 2 or faces.size(1) != 3:
        _err("faces must have dimensions (num_faces, 3)")
    if verts_color.dim() != 2 or verts_color.size(0) != verts.size(0) or verts_color.size(1) != 3:
        _err("vert_color must have dimensions (num_verts, 3)")
    if faces_opacity.dim() != 1 or faces_opacity.size(0) != faces.size(0):
        _err("face_opacity must have dimensions (num_faces)")
    _check_common(verts, faces, mv_mats, proj_mats, inv_mv_mats, inv_proj_mats, verts_depth, faces_intense, False)
    if tets.dim() != 2 or tets.size(1) != 4:
        _err("tets must have dimensions (num_tets, 4)")
    if face_tets.dim() != 2 or face_tets.size(0) != faces.size(0) or face_tets.size(1) != 2:
        _err("face_tets must have dimensions (num_faces, 2)")
    if tet_faces.dim() != 2 or tet_faces.size(0) != tets.size(0) or tet_faces.size(1) != 4:
        _err("tet_faces must have dimensions (num_tets, 4)")
    _require_cuda(background, verts, faces, verts_color, faces_opacity, mv_mats, proj_mats, inv_mv_mats, inv_proj_mats,
                  verts_depth, faces_intense, tets, face_tets, tet_faces)
    lib = _lib.load()
    B, P, F, T = mv_mats.size(0), verts.size(0), faces.size(0), tets.size(0)
    H, W = int(image_height), int(image_width)
    dev = verts.device
    with _on_device(dev):
        u8 = dict(dtype=torch.uint8, device=dev)
        bg = _f32(background, "background")
        verts_c, faces_c = _f32(verts, "verts"), _i32(faces, "faces")
        vcol, fopa = _f32(verts_color, "verts_color"), _f32(faces_opacity, "faces_opacity")
        mv, pj = _f32(mv_mats, "mv_mats"), _f32(proj_mats, "proj_mats")
        imv, ipj = _f32(inv_mv_mats, "inv_mv_mats"), _f32(inv_proj_mats, "inv_proj_mats")
        fint = _f32(faces_intense, "faces_intense")
        _f32(verts_depth, "verts_depth")   # dtype check only: the tet renderer never reads it
        tets_c, ft_c, tf_c = _i32(tets, "tets"), _i32(face_tets, "face_tets"), _i32(tet_faces, "tet_faces")

        sizes = (ctypes.c_size_t * 3)()
        _lib.check(lib.dmr_tet_state_bytes(B, P, F, T, W, H, sizes))
        point_buf = torch.empty(sizes[0], **u8)
        face_buf = torch.empty(sizes[1], **u8)
        img_buf = torch.empty(sizes[2], **u8)
        out_color = torch.empty((B, NUM_CHANNELS, H, W), dtype=torch.float32, device=dev)
        out_depth = torch.empty((B, 1, H, W), dtype=torch.float32, device=dev)
        out_active = torch.empty((B, H, W), dtype=torch.float32, device=dev)

        tet_rec, rec_valid = _TetRecordCache.get(lib, (verts_c, faces_c, tets_c, ft_c, tf_c), T, dev)
        pinned = _Pinned.acquire(dev)
        _arm(pinned)
        stream = _stream()
        try:
            _lib.check(lib.dmr_tet_forward_bin(B, P, F, T, W, H, _ptr(verts_c), _ptr(faces_c), _ptr(vcol), _ptr(fopa),
                                               _ptr(mv), _ptr(pj), _ptr(tets_c), _ptr(ft_c), _ptr(tf_c), _ptr(point_buf),
                                               _ptr(face_buf), _ptr(tet_rec), rec_valid, pinned[2], stream))
            key = ("tet", B, P, F, T, W, H)
            spec, _cap = _speculative_binning(lib, key, u8)
            R, bin_buf = _wait_R(lib, pinned, key, spec, u8)
        finally:
            _Pinned.release(pinned)
        if inverses is not None:
            inverses.check()
        _lib.check(lib.dmr_tet_forward_render_views(B, P, F, T, W, H, R, int(ray_random_seed), int(first_view), _ptr(bg),
                                                    _ptr(mv), _ptr(pj), _ptr(imv), _ptr(ipj), _ptr(fint), _ptr(point_buf),
                                                    _ptr(face_buf), _ptr(tet_rec), _ptr(bin_buf), _ptr(img_buf),
                                                    _ptr(out_color), _ptr(out_depth), _ptr(out_active), stream))
        face_buf.tet_records = tet_rec     # kept alive (and found by render_tets_backward) through the face buffer
    return out_color, out_depth, out_active, point_buf, face_buf, bin_buf, img_buf


def render_tets_backward(background, verts, faces, verts_color, faces_opacity, mv_mats, proj_mats, inv_mv_mats,
                         inv_proj_mats, verts_depth, faces_intense, tets, face_tets, tet_faces, grad_color, grad_depth,
                         pointBuffer, faceBuffer, binningBuffer, imageBuffer, ray_random_seed=None, deterministic=False,
                         tet_records=None, camera_grads=False, vertex_grads=False, intensity_grads=False,
                         accumulate_into=None, dL_dout_alpha=None, background_grad=False):
    """RenderFTetsBackwardCUDA (render.cu:338-412).
    Returns (dL_dverts_color[P,3], dL_dfaces_opacity[F]).  `ray_random_seed` is an
    optional trailing argument beyond the reference's 20: the autograd wrapper passes
    the forward's seed so that jittered rays (seed > 0) are re-read from the image
    buffer; with the reference's 20 arguments pixel-centre rays are used.  `deterministic`: run-to-run reproducible
    gradients (dmr_tet_backward_deterministic).  `tet_records`: the adjacency records of the forward call (the
    autograd wrapper passes them; otherwise they are taken from the face buffer's attribute or rebuilt).
    `camera_grads`: also return dL_dmv_mats, dL_dproj_mats [B,4,4] (gradients with respect to the mv_mats / proj_mats
    tensors passed here, through the rays and the hit-point depth; dmr_tet_backward_camera) as two more elements.
    `vertex_grads`: also return dL_dverts [P,3] (gradient with respect to the vertex positions, through the (t, u, v)
    of every walked step; dmr_tet_backward_vertex) as the last element.
    `intensity_grads`: also return dL_dfaces_intense [B,F] (gradient with respect to the face intensities, through the
    colour of every walked step; dmr_tet_backward_intensity) as the last element, after dL_dverts when both are
    requested.
    `accumulate_into`: (dL_dverts_color, dL_dfaces_opacity, dL_dverts), existing contiguous fp32 tensors of shapes
    [P,3], [F], [P,3] that the gradients are ADDED to (and that are returned) instead of fresh zero tensors, in every
    mode.  dL_dverts may be None (a fresh tensor when vertex_grads is set); it is written only when vertex_grads is
    set.  The camera and intensity gradients are always fresh tensors.
    `dL_dout_alpha`: cotangent [B,1,H,W] of the alpha image (tet_alpha); it changes dL_dfaces_opacity only
    (dmr_tet_backward_alpha, in every mode above).
    `background_grad`: also return dL_dbackground, float32 [3], as the last element (dmr_tet_background_grad)."""
    lib = _lib.load()
    B, P, F, T = mv_mats.size(0), verts.size(0), faces.size(0), tets.size(0)
    H, W = grad_color.size(2), grad_color.size(3)
    dev = verts.device
    if ray_random_seed is None:
        ray_random_seed = 0
    into = (None, None, None)
    if accumulate_into is not None:
        into = tuple(accumulate_into)
        if len(into) != 3 or into[0] is None or into[1] is None:
            _err("accumulate_into must be (dL_dverts_color, dL_dfaces_opacity, dL_dverts or None)")
    for t, shape, n in zip(into, ((P, 3), (F,), (P, 3)), ("dL_dverts_color", "dL_dfaces_opacity", "dL_dverts")):
        if t is not None and (t.dtype != torch.float32 or not t.is_contiguous() or tuple(t.shape) != shape or
                              t.device != dev):
            _err("accumulate_into: %s must be a contiguous float32 %s tensor on %s" % (n, list(shape), dev))
    with _on_device(dev):
        z = dict(dtype=torch.float32, device=dev)
        dL_dverts_color = into[0] if into[0] is not None else torch.zeros((P, 3), **z)
        dL_dfaces_opacity = into[1] if into[1] is not None else torch.zeros((F,), **z)
        # [B,16] column-major = [B,4,4] gradients of the (column-major, i.e. transposed) matrix tensors given here
        cam = torch.zeros((2, B, 4, 4), **z) if camera_grads else None
        dL_dverts = (into[2] if into[2] is not None else torch.zeros((P, 3), **z)) if vertex_grads else None
        dL_dfint = torch.zeros((B, F), **z) if intensity_grads else None
        if B * H * W > 0 and F > 0 and T > 0:
            bg = _f32(background, "background")
            mv, pj = _f32(mv_mats, "mv_mats"), _f32(proj_mats, "proj_mats")
            imv, ipj = _f32(inv_mv_mats, "inv_mv_mats"), _f32(inv_proj_mats, "inv_proj_mats")
            fint = _f32(faces_intense, "faces_intense")
            gc, gd = _f32(grad_color, "grad_color"), _f32(grad_depth, "grad_depth")
            tet_rec = tet_records if tet_records is not None else getattr(faceBuffer, "tet_records", None)
            if tet_rec is None:
                # the face buffer did not come straight from render_tets (e.g. unpacked from autograd's saved
                # tensors, which drops Python attributes): rebuild the view-independent records
                tet_rec = torch.empty(lib.dmr_tet_records_bytes(T), dtype=torch.uint8, device=dev)
                _lib.check(lib.dmr_tet_build_records(P, F, T, _ptr(_f32(verts, "verts")), _ptr(_i32(faces, "faces")),
                                                     _ptr(_i32(tets, "tets")), _ptr(_i32(face_tets, "face_tets")),
                                                     _ptr(_i32(tet_faces, "tet_faces")), _ptr(tet_rec), _stream()))
            a = (B, P, F, T, W, H, int(ray_random_seed), _ptr(bg), _ptr(mv), _ptr(pj), _ptr(imv), _ptr(ipj), _ptr(fint),
                 _ptr(pointBuffer), _ptr(faceBuffer), _ptr(tet_rec), _ptr(imageBuffer), _ptr(gc), _ptr(gd),
                 _ptr(dL_dverts_color), _ptr(dL_dfaces_opacity))
            if dL_dout_alpha is not None:
                det = int(bool(deterministic))
                ga = _f32(dL_dout_alpha, "dL_dout_alpha")
                if ga.numel() != B * H * W:
                    _err("dL_dout_alpha must have dimensions (batch_size, 1, H, W)")
                cm, vx = int(bool(camera_grads)), int(bool(vertex_grads))
                # the workspace of the mode it modifies
                nbytes = (lib.dmr_tet_backward_intensity_bytes(B, P, F, W, H, det, cm, vx) if intensity_grads else
                          lib.dmr_tet_backward_vertex_bytes(B, P, F, W, H, det, cm) if vertex_grads else
                          lib.dmr_tet_backward_camera_bytes(B, P, F, W, H, det) if camera_grads else
                          lib.dmr_tet_backward_deterministic_bytes(P, F) if det else
                          lib.dmr_tet_backward_workspace_bytes(P))
                ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
                null = ctypes.c_void_p(0)
                c = (_ptr(cam[0]), _ptr(cam[1])) if camera_grads else (null, null)
                dv = _ptr(dL_dverts) if vertex_grads else null
                fi = _ptr(dL_dfint) if intensity_grads else null
                _lib.check(lib.dmr_tet_backward_alpha(*a, det, *c, dv, fi, _ptr(ga), _ptr(ws), ws.numel(), _stream()))
            elif intensity_grads:
                det = int(bool(deterministic))
                ws = torch.empty(lib.dmr_tet_backward_intensity_bytes(B, P, F, W, H, det, int(bool(camera_grads)),
                                                                      int(bool(vertex_grads))),
                                 dtype=torch.uint8, device=dev)
                null = ctypes.c_void_p(0)
                c = (_ptr(cam[0]), _ptr(cam[1])) if camera_grads else (null, null)
                dv = _ptr(dL_dverts) if vertex_grads else null
                _lib.check(lib.dmr_tet_backward_intensity(*a, det, *c, dv, _ptr(dL_dfint), _ptr(ws), ws.numel(),
                                                          _stream()))
            elif vertex_grads:
                det = int(bool(deterministic))
                ws = torch.empty(lib.dmr_tet_backward_vertex_bytes(B, P, F, W, H, det, int(bool(camera_grads))),
                                 dtype=torch.uint8, device=dev)
                c = (_ptr(cam[0]), _ptr(cam[1])) if camera_grads else (ctypes.c_void_p(0), ctypes.c_void_p(0))
                _lib.check(lib.dmr_tet_backward_vertex(*a, det, *c, _ptr(dL_dverts), _ptr(ws), ws.numel(), _stream()))
            elif camera_grads:
                ws = torch.empty(lib.dmr_tet_backward_camera_bytes(B, P, F, W, H, int(bool(deterministic))),
                                 dtype=torch.uint8, device=dev)
                _lib.check(lib.dmr_tet_backward_camera(*a, int(bool(deterministic)), _ptr(cam[0]), _ptr(cam[1]), _ptr(ws),
                                                       ws.numel(), _stream()))
            elif deterministic:
                ws = torch.empty(lib.dmr_tet_backward_deterministic_bytes(P, F), dtype=torch.uint8, device=dev)
                _lib.check(lib.dmr_tet_backward_deterministic(*a, _ptr(ws), ws.numel(), _stream()))
            else:
                ws = torch.empty(lib.dmr_tet_backward_workspace_bytes(P), dtype=torch.uint8, device=dev)
                _lib.check(lib.dmr_tet_backward(*a, _ptr(ws), ws.numel(), _stream()))
    out = (dL_dverts_color, dL_dfaces_opacity)
    if camera_grads:
        out += (cam[0], cam[1])
    if vertex_grads:
        out += (dL_dverts,)
    if intensity_grads:
        out += (dL_dfint,)
    if background_grad:
        with _on_device(dev):
            out += (_background_grad(lib.dmr_tet_background_grad_bytes, lib.dmr_tet_background_grad, B, W, H, imageBuffer,
                                     grad_color, dev),)
    return out
