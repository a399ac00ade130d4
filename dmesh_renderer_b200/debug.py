"""Typed views into the opaque state buffers (dmr_debug_view) for parity checks."""
import ctypes

import numpy as np
import torch

from . import _lib

KINDS = {
    "verts_image": (0, np.float32, 4),
    "tiles_touched": (1, np.uint32, 1),
    "offsets": (2, np.uint32, 1),
    "depth_keys": (3, np.uint32, 1),
    "tile_keys_unsorted": (4, np.uint32, 1),
    "values_unsorted": (5, np.uint32, 1),
    "tile_keys_sorted": (6, np.uint32, 1),
    "values_sorted": (7, np.uint32, 1),
    "ranges": (8, np.uint32, 2),
    "n_contrib": (9, np.uint32, 1),
    "final_T": (10, np.float32, 1),
    "first_face": (11, np.int32, 1),
    "first_tet": (12, np.int32, 1),
    "face_order": (13, np.uint32, 1),
    "tet_jitter": (14, np.float32, 2),    # pixel coordinates of the rays; written only when ray_random_seed > 0
}
# The reference's 64-bit (tile | depth) keys.  The native path sorts FACES by depth and instances by tile
# id only (csrc/common.cuh: bin_faces / bin_instances), so it never materialises them; they are recomposed
# here from the tile ids, the face ids and the per-(view, face) depth keys for the bit-exact parity checks.
COMPOSED = {"keys_unsorted": ("tile_keys_unsorted", "values_unsorted"), "keys_sorted": ("tile_keys_sorted", "values_sorted")}


def view(renderer, kind, buffer, B, P, F, W, H, R=0, T=0, face_buffer=None):
    """Return a numpy copy of one intermediate.  renderer: "tri" | "tet".
    keys_sorted / keys_unsorted additionally need the face buffer (depth keys)."""
    if kind in COMPOSED:
        if face_buffer is None:
            raise ValueError("%s is recomposed from tile ids and depth keys: pass face_buffer=" % kind)
        dims = dict(B=B, P=P, F=F, W=W, H=H, R=R, T=T)
        tile = view(renderer, COMPOSED[kind][0], buffer, **dims).astype(np.uint64)
        fid = view(renderer, COMPOSED[kind][1], buffer, **dims).astype(np.int64)
        depth = view(renderer, "depth_keys", face_buffer, **dims).astype(np.uint64)
        tiles_per_view = ((W + 15) // 16) * ((H + 15) // 16)
        b = (tile // np.uint64(tiles_per_view)).astype(np.int64)
        return (tile << np.uint64(32)) | depth[b * F + fid]
    lib = _lib.load()
    k, dtype, width = KINDS[kind]
    ptr = ctypes.c_void_p()
    cnt = ctypes.c_size_t()
    _lib.check(lib.dmr_debug_view(0 if renderer == "tri" else 1, k, B, P, F, T, W, H, R,
                                  ctypes.c_void_p(buffer.data_ptr()), ctypes.byref(ptr), ctypes.byref(cnt)))
    n = cnt.value
    if n == 0:
        return np.zeros((0, width) if width > 1 else (0,), dtype=dtype)
    off = ptr.value - buffer.data_ptr()
    nbytes = n * width * np.dtype(dtype).itemsize
    arr = buffer[off:off + nbytes].cpu().numpy().view(dtype)
    return arr.reshape(n, width) if width > 1 else arr


_TORCH_DTYPE = {np.float32: torch.float32, np.uint32: torch.int32, np.int32: torch.int32}


def view_torch(renderer, kind, buffer, B, P, F, W, H, R=0, T=0, face_buffer=None):
    """Like view(), but a torch tensor ON THE DEVICE aliasing the state buffer (no copy; uint32 data comes back as
    int32 bit patterns, the recomposed 64-bit keys as int64) -- for parity checks at sizes where host copies of
    every intermediate would dominate the test time (C4, C5)."""
    if kind in COMPOSED:
        if face_buffer is None:
            raise ValueError("%s is recomposed from tile ids and depth keys: pass face_buffer=" % kind)
        dims = dict(B=B, P=P, F=F, W=W, H=H, R=R, T=T)
        tile = view_torch(renderer, COMPOSED[kind][0], buffer, **dims).to(torch.int64)
        fid = view_torch(renderer, COMPOSED[kind][1], buffer, **dims).to(torch.int64)
        depth = view_torch(renderer, "depth_keys", face_buffer, **dims).to(torch.int64) & 0xffffffff
        tiles_per_view = ((W + 15) // 16) * ((H + 15) // 16)
        b = tile // tiles_per_view
        return (tile << 32) | depth[b * F + fid]
    lib = _lib.load()
    k, dtype, width = KINDS[kind]
    ptr = ctypes.c_void_p()
    cnt = ctypes.c_size_t()
    _lib.check(lib.dmr_debug_view(0 if renderer == "tri" else 1, k, B, P, F, T, W, H, R,
                                  ctypes.c_void_p(buffer.data_ptr()), ctypes.byref(ptr), ctypes.byref(cnt)))
    n = cnt.value
    tdt = _TORCH_DTYPE[dtype]
    if n == 0:
        return torch.zeros((0, width) if width > 1 else (0,), dtype=tdt, device=buffer.device)
    off = ptr.value - buffer.data_ptr()
    t = buffer[off:off + n * width * 4].view(tdt)
    return t.view(n, width) if width > 1 else t
