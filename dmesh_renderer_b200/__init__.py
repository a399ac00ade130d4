"""dmesh_renderer_b200 -- B200-native drop-in for the `dmesh_renderer` package.

Public surface = the reference's (/root/reference/dmesh_renderer/__init__.py):
    TriRenderSettings, render_tri, TriRenderer          (:13-225)
    TetRenderSettings, render_tet, TetRenderer          (:237-488)
with identical argument order, dtype handling, return values and gradient
positions.  `import dmesh_renderer_b200 as dmesh_renderer` is the whole
migration (see INTEGRATION.md).

All compute runs in hand-written sm_100a CUDA kernels behind the C ABI of
libdmesh_b200.so (include/dmesh_b200.h) through the `_C` shim; PyTorch provides
device memory, the current stream and autograd plumbing only.
"""
from typing import NamedTuple

import torch as th

from . import _C

__all__ = ["TriRenderSettings", "render_tri", "TriRenderer", "TetRenderSettings", "render_tet", "TetRenderer"]


# =============================================================================
# TriRenderer: semi-transparent triangles, mean-depth ordered compositing.
# =============================================================================
class TriRenderSettings(NamedTuple):      # reference __init__.py:13-16
    image_height: int
    image_width: int
    bg: th.Tensor


_deterministic_default = False


def set_deterministic(flag: bool) -> bool:
    """Process-wide default for the backward passes of both renderers (extension, SURVEY.md 8f-3): True = run-to-run
    reproducible gradients (64-bit fixed-point accumulation instead of fp32 atomics; same values within fp32
    accumulation noise, slower).  `TriRenderer(settings, deterministic=...)` / `render_tri(..., deterministic=...)`
    override it per renderer / call (TetRenderer / render_tet likewise).  Returns the previous value."""
    global _deterministic_default
    old, _deterministic_default = _deterministic_default, bool(flag)
    return old


_exact_vertex_grads_default = False


def set_exact_vertex_grads(flag: bool) -> bool:
    """Process-wide default for the tri renderer's vertex-position gradient (extension).  False (the default): the
    reference implementation's formula, which differentiates the ray parameter t where the forward pass uses the
    second barycentric v.  True: the exact derivative of the rendered image, consistent with the camera gradients.
    The other gradients are the same either way.  `TriRenderer(settings, exact_vertex_grads=...)` /
    `render_tri(..., exact_vertex_grads=...)` override it per renderer / call.  Returns the previous value."""
    global _exact_vertex_grads_default
    old, _exact_vertex_grads_default = _exact_vertex_grads_default, bool(flag)
    return old


def render_tri(verts, faces, verts_color, faces_opacity, mv_mats, proj_mats, verts_depth, faces_intense,
               render_settings: TriRenderSettings, deterministic=None, exact_vertex_grads=None, return_alpha=False,
               return_face_weights=False):
    """reference __init__.py:18-43 (`deterministic`: see set_deterministic; `exact_vertex_grads`: see
    set_exact_vertex_grads; `return_alpha`, `return_face_weights`: see TriRenderer.forward).  render_settings.bg is
    passed to autograd as an input of its own: with bg.requires_grad set it gets its gradient."""
    det = _deterministic_default if deterministic is None else bool(deterministic)
    exact = _exact_vertex_grads_default if exact_vertex_grads is None else bool(exact_vertex_grads)
    return _RenderTri.apply(verts, faces, verts_color, faces_opacity, mv_mats, proj_mats, verts_depth, faces_intense,
                            render_settings, det, exact, bool(return_alpha), render_settings.bg,
                            bool(return_face_weights))


def _bg_for_render(bg):
    """The background the kernels read: unchanged unless it takes a gradient, then a detached fp32 copy (so a
    float64 leaf can be optimised; its gradient is returned in its own dtype)."""
    return bg.detach().to(th.float32) if bg.requires_grad else bg


class _RenderTri(th.autograd.Function):
    """reference __init__.py:45-170"""

    @staticmethod
    def forward(ctx, verts, faces, verts_color, faces_opacity, mv_mats, proj_mats, verts_depth, faces_intense,
                render_settings, deterministic=False, exact_vertex_grads=False, return_alpha=False, bg=None,
                return_face_weights=False):
        ctx.deterministic = deterministic
        ctx.exact_vertex_grads = exact_vertex_grads
        ctx.return_alpha = return_alpha
        bg = render_settings.bg if bg is None else bg
        ctx.bg_meta = (bg.dtype, bg.shape)
        bg = _bg_for_render(bg)
        try:
            # Same computation as _C.render_tris(*13 args) (reference __init__.py:62-88), issued in two halves
            # (phase 1: preprocess + scan; phase 2 after the num_rendered read-back).
            # depth in [-1, 1]: -1 near, 1 far
            inv = _C._Inverses(mv_mats, proj_mats)   # th.inverse x2 (reference :62-63): one launch, no device sync
            inv_mv_mats, inv_proj_mats = inv.inv_mv, inv.inv_proj
            mv_mats, proj_mats = inv.mv, inv.proj    # contiguous copies written by the same launch
            pending = _C.tri_forward_begin(bg, verts, faces, verts_color, faces_opacity, mv_mats,
                                           proj_mats, verts_depth, faces_intense, render_settings.image_height,
                                           render_settings.image_width)
            # speculative: phase 2 is enqueued before num_rendered reaches the host; `num_rendered` is then the count
            # the binning buffer was laid out for (>= the real one), which is what backward needs
            out = _C.tri_forward_finish(pending, inv_mv_mats, inv_proj_mats, inv, speculative=True,
                                        face_weights=return_face_weights)
            num_rendered, color, depth, pointBuffer, faceBuffer, binningBuffer, imgBuffer = out[:7]
        except Exception as ex:
            print("\nAn error occured in forward.")
            print(ex)
            raise ex
        ctx.render_settings = render_settings
        ctx.bg = bg
        ctx.num_rendered = num_rendered
        ctx.fused_depth = verts_depth is None
        ctx.grad_sink = _C.grad_sink_for(verts, verts_color, faces_opacity)   # multiview.PackedSceneGrads.direct()
        ctx.save_for_backward(verts, faces, verts_color, faces_opacity, mv_mats, proj_mats, inv_mv_mats, inv_proj_mats,
                              verts_depth, faces_intense, pointBuffer, faceBuffer, binningBuffer, imgBuffer)
        res = (color, depth)
        if return_alpha:
            # alpha = 1 - final_T, read from the image state after phase 2 (zeros when P == 0)
            res += (_C.tri_alpha(imgBuffer, color.size(0), color.size(2), color.size(3), color.device),)
        if return_face_weights:
            # face_weights, face_hits: statistics of phase 2, no gradient
            ctx.mark_non_differentiable(*out[7:])
            res += tuple(out[7:])
        return res

    @staticmethod
    def backward(ctx, grad_out_color, grad_out_depth, *grad_rest):
        # grad_rest: the alpha cotangent (return_alpha), then those of the face statistics (ignored)
        grad_out_alpha = grad_rest[0] if ctx.return_alpha else None
        num_rendered = ctx.num_rendered
        (verts, faces, verts_color, faces_opacity, mv_mats, proj_mats, inv_mv_mats, inv_proj_mats, verts_depth,
         faces_intense, pointBuffer, faceBuffer, binningBuffer, imgBuffer) = ctx.saved_tensors
        args = (ctx.bg, verts, faces, verts_color, faces_opacity, mv_mats, proj_mats, inv_mv_mats,
                inv_proj_mats, verts_depth, faces_intense, grad_out_color, grad_out_depth, num_rendered, pointBuffer,
                faceBuffer, binningBuffer, imgBuffer)
        sink = ctx.grad_sink
        into = None
        if sink is not None and sink.bind() == 0:
            into = tuple(leaf.grad for leaf in sink.leaves)
        # (bind() != 0: a leaf's .grad was dropped or replaced between forward and backward -- e.g. zero_grad with
        # set_to_none=True; the sink has re-attached it and this call hands its gradients to autograd the ordinary way)
        # camera gradients (extension): requested by setting requires_grad on mv_mats or proj_mats; they are per view and
        # always go through autograd (never into a gradient sink)
        camera = ctx.needs_input_grad[4] or ctx.needs_input_grad[5]
        # background gradient (extension): requested by setting requires_grad on render_settings.bg
        background = ctx.needs_input_grad[12]
        grad_mv = grad_proj = grad_bg = None
        try:
            grads = _C.render_tris_backward(*args, accumulate_into=into, deterministic=ctx.deterministic,
                                            camera_grads=camera, exact_vertex_grads=ctx.exact_vertex_grads,
                                            dL_dout_alpha=grad_out_alpha if ctx.return_alpha else None,
                                            background_grad=background)
        except Exception as ex:
            print("\nAn error occured in backward.\n")
            raise ex
        grad_verts, grad_verts_color, grad_faces_opacity, grad_verts_depth, grad_faces_intense = grads[:5]
        if camera:
            grad_mv, grad_proj = grads[5], grads[6]
        if background:
            grad_bg = grads[-1].to(ctx.bg_meta[0]).view(ctx.bg_meta[1])
        if ctx.fused_depth:
            # verts_depth=None: the depth was the vertex's own NDC z -> chain its gradient into the vertex positions
            # (and, for camera gradients, into the matrices)
            _C.tri_depth_chain(verts, mv_mats, proj_mats, grad_verts_depth, grad_verts, grad_mv, grad_proj)
            grad_verts_depth = None
        if into is not None:
            # already added to the leaves' .grad by the kernels
            grad_verts = grad_verts_color = grad_faces_opacity = None
        # gradient positions: reference __init__.py:156-168; positions 4 and 5 (the matrices) and 12 (bg) are an
        # extension
        return (grad_verts, None, grad_verts_color, grad_faces_opacity,
                grad_mv if ctx.needs_input_grad[4] else None, grad_proj if ctx.needs_input_grad[5] else None,
                grad_verts_depth, grad_faces_intense, None, None, None, None, grad_bg, None)


class TriRenderer(th.nn.Module):
    """reference __init__.py:172-225"""

    def __init__(self, render_settings: TriRenderSettings, deterministic=None, exact_vertex_grads=None,
                 return_alpha=False, return_face_weights=False):
        super().__init__()
        self.render_settings = render_settings
        self.deterministic = deterministic     # None: the process-wide default (set_deterministic)
        self.exact_vertex_grads = exact_vertex_grads   # None: the process-wide default (set_exact_vertex_grads)
        self.return_alpha = bool(return_alpha)
        self.return_face_weights = bool(return_face_weights)

    def forward(self, verts, faces, verts_color, faces_opacity, mv_mats, proj_mats, verts_depth, faces_intense):
        """
        verts [P,3] f32, faces [F,3] int, verts_color [P,3], faces_opacity [F]   (view independent)
        mv_mats, proj_mats [B,4,4] in maths convention (transposed here, as the reference does)
        verts_depth [B,P], faces_intense [B,F]                                   (per view)
        verts_depth=None (extension): use each vertex's own NDC z, computed and differentiated inside the
        renderer (what DMesh's callers otherwise compute upstream in PyTorch, a [B,P] tensor per step)
        returns color [B,3,H,W], depth [B,1,H,W]
        return_alpha (extension): also return alpha [B,1,H,W] fp32, differentiable: 1 - the transmittance the
        background was multiplied by (zeros when there are no vertices), for mask / silhouette losses.  Its gradient
        reaches faces_opacity only.  render_settings.bg gets a gradient when it requires grad.
        return_face_weights (extension): also return face_weights [B,F] fp32 and face_hits [B,F] int32, last, without
        gradient: per view, the sum over the pixels where a face was composited of T * alpha -- the factor its colour
        was multiplied by -- and the number of those pixels (for pruning, finding unseen faces, refinement).  Summed
        over faces, face_weights[b] equals alpha[b].sum() up to fp32 rounding.  Weights are accumulated in 64-bit fixed
        point with 32 fractional bits, so the statistics are bit-identical from run to run in both modes, and a weight
        below 2^-33 adds 0 (face_hits > 0 with face_weights == 0 is possible).  Images and gradients are unchanged.
        """
        return render_tri(verts, faces.to(dtype=th.int32), verts_color, faces_opacity, mv_mats.transpose(1, 2),
                          proj_mats.transpose(1, 2), verts_depth, faces_intense, self.render_settings,
                          self.deterministic, self.exact_vertex_grads, self.return_alpha, self.return_face_weights)


# =============================================================================
# TetRenderer: faces of a tetrahedral complex, exact depth order by ray marching
# through tet adjacency; gradients to vertex colours, face opacities and (opt-in) the camera matrices, the
# vertex positions and the face intensities.
# =============================================================================
class TetRenderSettings(NamedTuple):      # reference __init__.py:237-241
    image_height: int
    image_width: int
    bg: th.Tensor
    ray_random_seed: int


_tet_vertex_grads_default = False


def set_tet_vertex_grads(flag: bool) -> bool:
    """Process-wide default for the tet renderer's vertex-position gradient (extension).  False (the default): like the
    reference, the tet renderer returns no gradient for verts.  True: when verts requires grad, its gradient is the
    exact derivative of the rendered colour and depth images, consistent with the camera gradients.  The other
    gradients are the same either way.  `TetRenderer(settings, vertex_grads=...)` / `render_tet(..., vertex_grads=...)`
    override it per renderer / call.  Returns the previous value."""
    global _tet_vertex_grads_default
    old, _tet_vertex_grads_default = _tet_vertex_grads_default, bool(flag)
    return old


_tet_intensity_grads_default = False


def set_tet_intensity_grads(flag: bool) -> bool:
    """Process-wide default for the tet renderer's face-intensity gradient (extension).  False (the default): like the
    reference, the tet renderer returns no gradient for faces_intense.  True: when faces_intense requires grad, its
    gradient is the exact derivative of the rendered colour image (depth does not depend on it).  The other gradients
    are the same either way.  `TetRenderer(settings, intensity_grads=...)` / `render_tet(..., intensity_grads=...)`
    override it per renderer / call.  Returns the previous value."""
    global _tet_intensity_grads_default
    old, _tet_intensity_grads_default = _tet_intensity_grads_default, bool(flag)
    return old


def render_tet(verts, faces, verts_color, faces_opacity, mv_mats, proj_mats, verts_depth, faces_intense, tets,
               face_tets, tet_faces, render_settings: TetRenderSettings, deterministic=None, vertex_grads=None,
               intensity_grads=None, first_view=0, return_alpha=False, return_face_weights=False):
    """reference __init__.py:243-275 (`deterministic`: see set_deterministic; `vertex_grads`: see
    set_tet_vertex_grads; `intensity_grads`: see set_tet_intensity_grads; `first_view`, `return_alpha`,
    `return_face_weights`: see TetRenderer.forward).  render_settings.bg is passed to autograd as an input of its own: with bg.requires_grad set
    it gets its gradient."""
    det = _deterministic_default if deterministic is None else bool(deterministic)
    vert = _tet_vertex_grads_default if vertex_grads is None else bool(vertex_grads)
    fint = _tet_intensity_grads_default if intensity_grads is None else bool(intensity_grads)
    return _RenderTet.apply(verts, faces, verts_color, faces_opacity, mv_mats, proj_mats, verts_depth, faces_intense,
                            tets, face_tets, tet_faces, render_settings, det, vert, fint, int(first_view),
                            bool(return_alpha), render_settings.bg, bool(return_face_weights))


class _RenderTet(th.autograd.Function):
    """reference __init__.py:277-424"""

    @staticmethod
    def forward(ctx, verts, faces, verts_color, faces_opacity, mv_mats, proj_mats, verts_depth, faces_intense, tets,
                face_tets, tet_faces, render_settings, deterministic=False, vertex_grads=False, intensity_grads=False,
                first_view=0, return_alpha=False, bg=None, return_face_weights=False):
        ctx.deterministic = deterministic
        ctx.vertex_grads = vertex_grads
        ctx.intensity_grads = intensity_grads
        ctx.return_alpha = return_alpha
        bg = render_settings.bg if bg is None else bg
        ctx.bg_meta = (bg.dtype, bg.shape)
        bg = ctx.bg = _bg_for_render(bg)
        inv = _C._Inverses(mv_mats, proj_mats)   # th.inverse x2 (reference :298-299): one launch, no device sync
        inv_mv_mats, inv_proj_mats = inv.inv_mv, inv.inv_proj
        mv_mats, proj_mats = inv.mv, inv.proj    # contiguous copies written by the same launch
        args = (bg, verts, faces, verts_color, faces_opacity, mv_mats, proj_mats, inv_mv_mats,
                inv_proj_mats, verts_depth, faces_intense, tets, face_tets, tet_faces, render_settings.image_height,
                render_settings.image_width, render_settings.ray_random_seed, inv)
        try:
            color, depth, active, pointBuffer, faceBuffer, binningBuffer, imgBuffer = _C.render_tets(
                *args, first_view=first_view)
        except Exception as ex:
            print("\nAn error occured in forward.")
            raise ex
        active = (active > 0.5)
        ctx.render_settings = render_settings
        ctx.tet_records = getattr(faceBuffer, "tet_records", None)   # cached adjacency records (no gradient, not an input)
        ctx.grad_sink = _C.grad_sink_for(verts, verts_color, faces_opacity, tet=True)   # PackedSceneGrads.direct()
        ctx.save_for_backward(verts, faces, verts_color, faces_opacity, mv_mats, proj_mats, inv_mv_mats, inv_proj_mats,
                              verts_depth, faces_intense, tets, face_tets, tet_faces, pointBuffer, faceBuffer,
                              binningBuffer, imgBuffer)
        ctx.mark_non_differentiable(active)
        res = (color, depth, active)
        if return_alpha:
            res += (_C.tet_alpha(imgBuffer, color.size(0), color.size(2), color.size(3), color.device),)
        if return_face_weights:
            # face_weights, face_hits: a post-pass over the forward state, no gradient
            stats = _C.tet_face_weights(color.size(0), verts.size(0), faces.size(0), tets.size(0), color.size(2),
                                        color.size(3), render_settings.ray_random_seed, inv_mv_mats, inv_proj_mats,
                                        pointBuffer, faceBuffer, imgBuffer, ctx.tet_records)
            ctx.mark_non_differentiable(*stats)
            res += stats
        return res

    @staticmethod
    def backward(ctx, grad_out_color, grad_out_depth, grad_out_active, *grad_rest):
        # grad_rest: the alpha cotangent (return_alpha), then those of the face statistics (ignored)
        grad_out_alpha = grad_rest[0] if ctx.return_alpha else None
        render_settings = ctx.render_settings
        (verts, faces, verts_color, faces_opacity, mv_mats, proj_mats, inv_mv_mats, inv_proj_mats, verts_depth,
         faces_intense, tets, face_tets, tet_faces, pointBuffer, faceBuffer, binningBuffer, imgBuffer) = ctx.saved_tensors
        args = (ctx.bg, verts, faces, verts_color, faces_opacity, mv_mats, proj_mats, inv_mv_mats,
                inv_proj_mats, verts_depth, faces_intense, tets, face_tets, tet_faces, grad_out_color, grad_out_depth,
                pointBuffer, faceBuffer, binningBuffer, imgBuffer, render_settings.ray_random_seed)
        # camera gradients (extension): requested by setting requires_grad on mv_mats or proj_mats; per view, through
        # autograd only
        camera = ctx.needs_input_grad[4] or ctx.needs_input_grad[5]
        # vertex-position gradients (extension): only when switched on AND verts requires grad (DMesh passes verts
        # that require grad, so requires_grad alone must not turn this on)
        vertex = ctx.vertex_grads and ctx.needs_input_grad[0]
        # face-intensity gradients (extension): likewise only when switched on AND faces_intense requires grad (callers
        # compute intensities from verts, e.g. a Lambertian term)
        intensity = ctx.intensity_grads and ctx.needs_input_grad[7]
        # background gradient (extension): requested by setting requires_grad on render_settings.bg
        background = ctx.needs_input_grad[17]
        grad_mv = grad_proj = grad_verts = grad_fint = grad_bg = None
        # a gradient sink takes verts_color, faces_opacity and, when it has a verts slot and the vertex-position path
        # runs, verts; camera and intensity gradients are per view and always go through autograd
        sink = ctx.grad_sink
        into = None
        if sink is not None and sink.bind() == 0:   # (bind() != 0: see _RenderTri.backward)
            g = [leaf.grad for leaf in sink.leaves]
            into = (g[-2], g[-1], g[0] if len(g) == 3 and vertex else None)
        try:
            grads = _C.render_tets_backward(*args, deterministic=ctx.deterministic, tet_records=ctx.tet_records,
                                            camera_grads=camera, vertex_grads=vertex, intensity_grads=intensity,
                                            accumulate_into=into,
                                            dL_dout_alpha=grad_out_alpha if ctx.return_alpha else None,
                                            background_grad=background)
        except Exception as ex:
            print("\nAn error occured in backward.\n")
            raise ex
        grad_verts_color, grad_faces_opacity = grads[:2]
        if background:
            grad_bg = grads[-1].to(ctx.bg_meta[0]).view(ctx.bg_meta[1])
            grads = grads[:-1]
        if camera:
            grad_mv, grad_proj = grads[2], grads[3]
        if intensity:
            grad_fint = grads[-1]
        if vertex:
            grad_verts = grads[-2] if intensity else grads[-1]
        if into is not None:
            # already added to the leaves' .grad by the kernels
            grad_verts_color = grad_faces_opacity = None
            if into[2] is not None:
                grad_verts = None
        # gradient positions: reference __init__.py:407-422; positions 0 (verts), 4, 5 (the matrices), 7
        # (faces_intense) and 17 (bg) are an extension
        return (grad_verts, None, grad_verts_color, grad_faces_opacity,
                grad_mv if ctx.needs_input_grad[4] else None, grad_proj if ctx.needs_input_grad[5] else None,
                None, grad_fint, None, None, None, None, None, None, None, None, None, grad_bg, None)


class TetRenderer(th.nn.Module):
    """reference __init__.py:426-488"""

    def __init__(self, render_settings: TetRenderSettings, deterministic=None, vertex_grads=None, intensity_grads=None,
                 return_alpha=False, return_face_weights=False):
        super().__init__()
        self.render_settings = render_settings
        self.return_alpha = bool(return_alpha)
        self.return_face_weights = bool(return_face_weights)
        self.deterministic = deterministic     # None: the process-wide default (set_deterministic)
        self.vertex_grads = vertex_grads       # None: the process-wide default (set_tet_vertex_grads)
        self.intensity_grads = intensity_grads   # None: the process-wide default (set_tet_intensity_grads)

    def forward(self, verts, faces, verts_color, faces_opacity, mv_mats, proj_mats, verts_depth, faces_intense, tets,
                face_tets, tet_faces, first_view=0):
        """
        Gradients for verts_color and faces_opacity, and (extension) for mv_mats / proj_mats when they require
        grad, for verts when vertex_grads is on and verts requires grad, and for faces_intense when intensity_grads
        is on and faces_intense requires grad (returned in faces_intense's own dtype and shape, e.g. float64 or a
        stride-0 expanded [B,F]).  verts_depth is accepted but unused (depth comes from the re-projected hit point).
        tets [T,4], face_tets [F,2] (-1 = boundary), tet_faces [T,4]
        first_view (extension): index of view 0 of this call in a larger job, e.g. a rank's share of the cameras
        (multiview.shard_views(...).start).  With ray_random_seed > 0 the jittered rays of a view then depend only on
        its index in the job, so rendering views s..e-1 with first_view=s gives exactly views s..e-1 of one call over
        all views.  0, the default, gives the reference's rays.
        returns color [B,3,H,W], depth [B,1,H,W], active [B,H,W] bool
        return_alpha (extension): also return alpha [B,1,H,W] fp32, differentiable: 1 - the transmittance the
        background was multiplied by on active pixels, 0 on inactive ones.  Its gradient reaches faces_opacity only.
        render_settings.bg gets a gradient when it requires grad.
        return_face_weights (extension): also return face_weights [B,F] fp32 and face_hits [B,F] int32, last, without
        gradient: per view, the sum over the active pixels where a face was composited of expf(log_T) * opacity -- the
        factor its colour was multiplied by -- and the number of those pixels.  Inactive pixels count for nothing.
        Summed over faces, face_weights[b] equals alpha[b].sum() up to fp32 rounding (not where a face of opacity 1
        ends a ray).  Same fixed-point format and reproducibility as TriRenderer's.  Computed by one post-pass over
        the forward state; images and gradients are unchanged.
        """
        f32, i32 = th.float32, th.int32
        return render_tet(verts.to(dtype=f32), faces.to(dtype=i32), verts_color.to(dtype=f32),
                          faces_opacity.to(dtype=f32), mv_mats.to(dtype=f32).transpose(1, 2),
                          proj_mats.to(dtype=f32).transpose(1, 2), verts_depth.to(dtype=f32),
                          faces_intense.to(dtype=f32), tets.to(dtype=i32), face_tets.to(dtype=i32),
                          tet_faces.to(dtype=i32), self.render_settings, self.deterministic, self.vertex_grads,
                          self.intensity_grads, first_view, self.return_alpha, self.return_face_weights)
