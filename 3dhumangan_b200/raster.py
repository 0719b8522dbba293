"""The preprocessor's mesh rasteriser on the device (SURVEY.md 8f-2): the segmentation targets of every training iteration.

The reference makes them in `SHHQPreprocessor._forward_rasterize` (lib/data/preprocessor.py:138-176) with pytorch3d's
`MeshRasterizer`; here one library call (csrc/raster.cu, `hg_mesh_raster`) rasterises the posed mesh and writes the label map
and the semantic map directly.

    pix_to_face, zbuf, bary = rasterize(verts [B,V,3], faces [F,3], R [B,3,3], T [B,3], focal, H, W)
    segments, semantics     = rasterize_labels(verts, faces, faces_to_labels [F], sem_verts [V,3], R, T, focal, H, W)

    pre = SHHQPreprocessor(gen_height, gen_width)      # lib/data/preprocessor.py:14-176, same buffers / state_dict
    pre.init_smpl(smpl_faces, smpl_faces_to_labels)    # from SMPL_NEUTRAL.pkl / densepose_data.json (the caller's)
    data = pre(data, rotate=True, **metadata)          # + cam2world_matrices, rasterized_segments, rasterized_semantics

Semantics: pytorch3d 0.6.2's MeshRasterizer with faces_per_pixel = 1, blur_radius = 0, no back-face culling,
perspective-correct barycentrics, cameras `PerspectiveCameras(in_ndc=True)` (view = X @ R + T), as restated in
oracle/raster_port.py (that restatement is unpinned against pytorch3d itself; see DESIGN.md section 2).  `pix_to_face` is
pytorch3d's packed index b * F + face with -1 for the background; `zbuf` and `bary` are -1 there.  Other settings, gradients
and `coordinate_mode='fix_camera'` raise RuntimeError; so does every entry without the library or a CUDA device.

Face indices are checked against V on the host once per face tensor (kept in a small cache with an int32 copy), so the first
call with a new face tensor synchronises; calls after it can be captured into a CUDA graph."""
from __future__ import annotations

import math

import torch
import torch.nn as nn

from . import abi, smpl

FOCAL_RASTER = 1.0 / math.tan(math.pi * 1 / 180 / 2)      # preprocessor.py:145-146 (the camera gets -FOCAL_RASTER)

_FACES = {}


def _faces_i32(faces, V, device):
    """Validated int32 copy of `faces` on `device` (cached; the cache keeps `faces` alive so its address is not reused)."""
    key = (faces.data_ptr(), faces._version, tuple(faces.shape), faces.dtype, str(faces.device), V, str(device))
    ent = _FACES.get(key)
    if ent is None:
        if faces.dim() != 2 or faces.shape[1] != 3 or faces.shape[0] == 0 or faces.dtype.is_floating_point:
            raise RuntimeError("hg3d raster: faces must be a non-empty integer tensor [F,3]")
        lo, hi = int(faces.min()), int(faces.max())
        if lo < 0 or hi >= V:
            raise RuntimeError(f"hg3d raster: face indices must lie in [0, {V}); got [{lo}, {hi}]")
        if len(_FACES) >= 16:
            _FACES.clear()
        ent = _FACES[key] = (faces, faces.to(device=device, dtype=torch.int32).contiguous())
    return ent[1]


def _check(verts, R, T, H, W, faces_per_pixel, blur_radius, cull_backfaces):
    abi.require_device()
    if faces_per_pixel != 1 or blur_radius != 0.0 or cull_backfaces:
        raise RuntimeError("hg3d raster: only faces_per_pixel=1, blur_radius=0, cull_backfaces=False (the preprocessor's settings)")
    if torch.is_grad_enabled() and verts.requires_grad:
        raise RuntimeError("hg3d raster: no gradients (the reference rasterises under no_grad)")
    if verts.dim() != 3 or verts.shape[2] != 3 or tuple(R.shape) != (verts.shape[0], 3, 3) or tuple(T.shape) != (verts.shape[0], 3):
        raise RuntimeError("hg3d raster: verts [B,V,3], R [B,3,3], T [B,3]")
    if not verts.is_cuda:
        raise RuntimeError("hg3d raster: expected CUDA tensors (there is no CPU path)")
    if H <= 0 or W <= 0:
        raise RuntimeError("hg3d raster: bad image size")


def _launch(verts, faces, R, T, focal, H, W, labels=None, sem_verts=None, p2f=False, zbuf=False, bary=False):
    dev = verts.device
    B, V = verts.shape[0], verts.shape[1]
    f32 = lambda t: t.to(device=dev, dtype=torch.float32).contiguous()
    verts, R, T = f32(verts), f32(R), f32(T)
    fi = _faces_i32(faces, V, dev)
    F = fi.shape[0]
    out = {}
    if p2f:
        out["pix_to_face"] = torch.empty(B, H, W, dtype=torch.int64, device=dev)
    if zbuf:
        out["zbuf"] = torch.empty(B, H, W, dtype=torch.float32, device=dev)
    if bary:
        out["bary"] = torch.empty(B, H, W, 3, dtype=torch.float32, device=dev)
    if labels is not None:
        if labels.shape != (F,):
            raise RuntimeError("hg3d raster: faces_to_labels must be [F]")
        labels = labels.to(device=dev, dtype=torch.int64).contiguous()
        out["segments"] = torch.empty(B, H, W, dtype=torch.int64, device=dev)
    if sem_verts is not None:
        if sem_verts.shape != (V, 3):
            raise RuntimeError("hg3d raster: sem_verts must be [V,3]")
        sem_verts = f32(sem_verts)
        out["semantics"] = torch.empty(B, 3, H, W, dtype=torch.float32, device=dev)
    keys = torch.empty(B, H, W, dtype=torch.int64, device=dev)
    with torch.cuda.device_of(verts):
        abi.call("hg_mesh_raster", abi.ptr(verts), abi.ptr(fi), abi.ptr(R), abi.ptr(T), float(focal), B, V, F, H, W, abi.ptr(keys),
                 abi.ptr(labels), abi.ptr(sem_verts), abi.ptr(out.get("pix_to_face")), abi.ptr(out.get("zbuf")),
                 abi.ptr(out.get("bary")), abi.ptr(out.get("segments")), abi.ptr(out.get("semantics")), abi.stream())
    return out


def rasterize(verts, faces, R, T, focal, H, W, *, faces_per_pixel=1, blur_radius=0.0, cull_backfaces=False):
    """pytorch3d's `MeshRasterizer(cameras=PerspectiveCameras(focal_length=focal, R=R, T=T, in_ndc=True))` over
    `Meshes(verts, faces shared by the batch)` with K = 1 squeezed -> (pix_to_face [B,H,W] int64 packed b*F + face,
    zbuf [B,H,W], bary [B,H,W,3]); background -1."""
    _check(verts, R, T, H, W, faces_per_pixel, blur_radius, cull_backfaces)
    o = _launch(verts, faces, R, T, focal, H, W, p2f=True, zbuf=True, bary=True)
    return o["pix_to_face"], o["zbuf"], o["bary"]


def rasterize_labels(verts, faces, faces_to_labels, sem_verts, R, T, focal, H, W):
    """preprocessor.py:152-174 fused: -> (segments [B,H,W] int64 = faces_to_labels[face] + 2, background 1;
    semantics [B,3,H,W] float32 = sem_verts at the face vertex with the largest barycentric, background 0)."""
    _check(verts, R, T, H, W, 1, 0.0, False)
    o = _launch(verts, faces, R, T, focal, H, W, labels=faces_to_labels, sem_verts=sem_verts)
    return o["segments"], o["semantics"]


class SHHQPreprocessor(nn.Module):
    """lib/data/preprocessor.py:14-176 on the device.  Same constructor, buffers (names, shapes, dtypes) and methods."""

    def __init__(self, gen_height, gen_width, **kwargs):
        super().__init__()
        self.height = gen_height
        self.width = gen_width
        self.mode = kwargs.get("coordinate_mode", "fix_body")
        if self.mode != "fix_body":
            raise RuntimeError(f"hg3d SHHQPreprocessor: coordinate_mode={self.mode!r} is not built (no shipped curriculum uses it)")
        self.register_buffer("vertex_approximation", torch.zeros([6890], dtype=torch.long))
        self.register_buffer("smpl_faces", torch.zeros([13776, 3], dtype=torch.long))
        self.register_buffer("smpl_faces_to_labels", torch.zeros([13776], dtype=torch.long))

    @torch.no_grad()
    def init_smpl(self, smpl_faces, smpl_faces_to_labels):
        smpl_faces = torch.as_tensor(smpl_faces)
        V = self.vertex_approximation.shape[0]
        if smpl_faces.numel() and (int(smpl_faces.min()) < 0 or int(smpl_faces.max()) >= V):
            raise RuntimeError(f"hg3d SHHQPreprocessor: face indices must lie in [0, {V})")
        self.smpl_faces.copy_(smpl_faces)
        self.smpl_faces_to_labels.copy_(torch.as_tensor(smpl_faces_to_labels))

    @torch.no_grad()
    def forward(self, data, rotate=False, **kwargs):
        batch_size = data["scales"].shape[0]
        h_rotation = torch.randn(batch_size) * (kwargs["h_stddev"] if rotate else 0) + kwargs["h_mean"]
        v_rotation = torch.randn(batch_size) * (kwargs["v_stddev"] if rotate else 0) + kwargs["v_mean"]
        r_rotation = torch.zeros_like(h_rotation)
        return self.forward_with_rotation(data, h_rotation, v_rotation, r_rotation, **kwargs)

    @torch.no_grad()
    def forward_with_rotation(self, data, h_rotation, v_rotation, r_rotation, **kwargs):
        """_forward_fix_body (cam2world_matrices, R_raster) + _forward_rasterize (rasterized_segments [B,H,W] int64,
        rasterized_semantics [B,3,H,W] float32); returns the mutated `data`."""
        abi.require_device()
        Rb = smpl.body_rotation(data, h_rotation, v_rotation, r_rotation)
        R_raster = torch.inverse(Rb)
        data["cam2world_matrices"] = smpl.cam2world_fix_body(data, h_rotation, v_rotation, r_rotation, Rb=Rb)
        T_raster = data["T"][:, :3, -1].clone()
        T_raster[:, -1] = FOCAL_RASTER / data["scales"] * 0.5
        seg, sem = rasterize_labels(data["vertices"], self.smpl_faces, self.smpl_faces_to_labels, data["tpose_vertices"][0],
                                    R_raster, T_raster, -FOCAL_RASTER, self.height, self.width)
        data["rasterized_semantics"] = sem
        data["rasterized_segments"] = seg
        return data
