"""Oracle for the preprocessor's mesh rasteriser (SURVEY.md 8f-2).  TEST INFRASTRUCTURE ONLY (imported by tests/ and
tests/golden/make_golden_raster.py).

`SHHQPreprocessor._forward_rasterize` (lib/data/preprocessor.py:138-176 of the reference) rasterises the posed SMPL mesh with
pytorch3d 0.6.2's `MeshRasterizer` (faces_per_pixel = 1, blur_radius = 0, no culling, perspective-correct barycentrics).
pytorch3d is not vendored and not installed, so its arithmetic is RESTATED here from its published `rasterize_meshes` /
`PerspectiveCameras` code with one fp32 IEEE operation per step, left to right, kEpsilon = 1e-8:

  view      Xv = ((X R00 + Y R10) + Z R20) + T0   (row vectors: X_world @ R + T), same for Yv, Zv
  NDC       xn = (f Xv) / Zv,  yn = (f Yv) / Zv,  z = Zv             (in_ndc PerspectiveCameras, principal point 0)
  pixel     x = PixToNonSquareNdc(W-1-xi, W, H), y = PixToNonSquareNdc(H-1-yi, H, W),
            PixToNonSquareNdc(i, S1, S2) = -o + (r i + o) / S1,  r = 2 (or (S1 * 2) / S2 if S1 > S2), o = r / 2
  reject    max(z0,z1,z2) < 0,  |E(v0,v1,v2)| <= eps,  pixel outside the face's closed xy box
            E(p,a,b) = (p.x-a.x)(b.y-a.y) - (p.y-a.y)(b.x-a.x)
  bary      area = E(v2,v0,v1) + eps, w0 = E(p,v1,v2)/area, w1 = E(p,v2,v0)/area, w2 = E(p,v0,v1)/area
  persp.    t0 = (w0 z1) z2, t1 = (z0 w1) z2, t2 = (z0 z1) w2, d = max((t0+t1)+t2, eps), wi = ti / d
  depth     pz = (w0 z0 + w1 z1) + w2 z2;  reject pz < 0;  inside iff w0 > 0 && w1 > 0 && w2 > 0
  z-buffer  smallest pz, lowest face index on equal pz (-0.0 == +0.0); background pix_to_face = zbuf = bary = -1

PINNING: the reference's own glue around the rasteriser (`_forward_fix_body`, `_forward_rasterize`) is pinned by
tests/golden/make_golden_raster.py, which runs those methods with the stand-ins below injected for pytorch3d's classes.  The
restatement itself is UNPINNED against pytorch3d (no copy of it exists here), exactly like `knn_points`.  The kernel
(csrc/raster.cu) reproduces this arithmetic bit for bit.

Everything is elementwise torch ops in the stated order (no matmul / einsum / bmm on values that decide coverage or depth:
GEMMs may contract or reorder), so the same functions run on the CPU and, as the GPU tests' checker, on the device.
Divisions are always tensor / tensor: CUDA torch turns a division by a Python scalar into a multiplication by its reciprocal."""
import math
from collections import namedtuple

import torch

from oracle.smpl_port import euler_xyz_to_matrix

K_EPSILON = 1e-8


def _ndc_params(S1, S2):
    """(r, o) of PixToNonSquareNdc in fp32."""
    r = torch.tensor(2.0, dtype=torch.float32)
    if S1 > S2:
        r = (torch.tensor(float(S1), dtype=torch.float32) * r) / torch.tensor(float(S2), dtype=torch.float32)
    return float(r), float(r / torch.tensor(2.0, dtype=torch.float32))


def _c(v, like):
    """A one-element tensor on `like`'s device and dtype (not a Python scalar: see the module docstring on division)."""
    return torch.full((1,), float(v), dtype=like.dtype, device=like.device)


def pix_to_ndc(i, S1, S2, like):
    """PixToNonSquareNdc for integer pixel indices `i` (a tensor), in the dtype of `like`."""
    r, o = _ndc_params(S1, S2)
    i = i.to(like.dtype)
    return (-_c(o, like)) + (_c(r, like) * i + _c(o, like)) / _c(S1, like)


def _edge(px, py, ax, ay, bx, by):
    return (px - ax) * (by - ay) - (py - ay) * (bx - ax)


def project(verts, R, T, focal):
    """verts [B,V,3], R [B,3,3], T [B,3], focal (scalar) -> xn, yn, z [B,V]."""
    X, Y, Z = verts[..., 0], verts[..., 1], verts[..., 2]
    r = lambda i, j: R[:, i, j][:, None]
    t = lambda i: T[:, i][:, None]
    Xv = ((X * r(0, 0) + Y * r(1, 0)) + Z * r(2, 0)) + t(0)
    Yv = ((X * r(0, 1) + Y * r(1, 1)) + Z * r(2, 1)) + t(1)
    Zv = ((X * r(0, 2) + Y * r(1, 2)) + Z * r(2, 2)) + t(2)
    f = _c(focal, verts)
    return (f * Xv) / Zv, (f * Yv) / Zv, Zv


def pixel_test(px, py, x0, y0, z0, x1, y1, z1, x2, y2, z2):
    """-> (covered, w0, w1, w2, pz) for pixel centres (px, py) against faces (all tensors of one shape); the face-level tests
    (zmax, zero area) are the caller's.  `covered` includes the closed-box test."""
    eps = _c(K_EPSILON, px)
    xmin, xmax = torch.fmin(torch.fmin(x0, x1), x2), torch.fmax(torch.fmax(x0, x1), x2)
    ymin, ymax = torch.fmin(torch.fmin(y0, y1), y2), torch.fmax(torch.fmax(y0, y1), y2)
    inbox = ~((px > xmax) | (px < xmin) | (py > ymax) | (py < ymin))
    area = _edge(x2, y2, x0, y0, x1, y1) + eps
    w0 = _edge(px, py, x1, y1, x2, y2) / area
    w1 = _edge(px, py, x2, y2, x0, y0) / area
    w2 = _edge(px, py, x0, y0, x1, y1) / area
    t0 = (w0 * z1) * z2
    t1 = (z0 * w1) * z2
    t2 = (z0 * z1) * w2
    d = torch.fmax((t0 + t1) + t2, eps)
    w0, w1, w2 = t0 / d, t1 / d, t2 / d
    pz = (w0 * z0 + w1 * z1) + w2 * z2
    covered = inbox & ~(pz < 0) & (w0 > 0) & (w1 > 0) & (w2 > 0)
    return covered, w0, w1, w2, pz


def _pixel_range(lo, hi, S1, S2):
    """Conservative (+-1 pixel) index range [i0, i1] of PixToNonSquareNdc covering [lo, hi]; non-finite -> the whole axis."""
    r, o = _ndc_params(S1, S2)
    lo64, hi64 = lo.double(), hi.double()
    finite = torch.isfinite(lo64) & torch.isfinite(hi64)
    i0 = torch.floor(((lo64.clamp(-1e6, 1e6) + o) * S1 - o) / r) - 1
    i1 = torch.ceil(((hi64.clamp(-1e6, 1e6) + o) * S1 - o) / r) + 1
    i0 = torch.where(finite, i0, torch.zeros_like(i0)).clamp(0, S1 - 1).long()
    i1 = torch.where(finite, i1, torch.full_like(i1, S1 - 1)).clamp(0, S1 - 1).long()
    return i0, i1


def depth_key(pz, face):
    """The z-buffer key (bits(pz) << 32) | face for pz >= 0 (fp32), -0.0 canonicalised to +0.0: orders like (pz, face)."""
    pz = torch.where(pz == 0, torch.zeros_like(pz), pz)
    return (pz.view(torch.int32).to(torch.int64) << 32) | face


def rasterize(verts, faces, R, T, focal, H, W, dtype=torch.float32):
    """-> pix_to_face [B,H,W] int64 (index into `faces`, -1 = background), zbuf [B,H,W], bary [B,H,W,3] in `dtype`.

    Vectorised over faces: each face's bounding-box pixels are enumerated, tested exactly, and the per-pixel minimum of
    key = (bits(pz) << 32) | face is taken with scatter_reduce (fp32); fp64 (an informational comparison only) takes the
    minimum pz, then the lowest face among the entries at that minimum."""
    dev = verts.device
    verts, R, T = verts.to(dtype), R.to(dtype), T.to(dtype)
    faces = faces.to(dev).long()
    B, F = verts.shape[0], faces.shape[0]
    xn, yn, zn = project(verts, R, T, focal)
    g = lambda a, k: a[:, faces[:, k]]                                      # [B,F]
    x0, y0, z0, x1, y1, z1, x2, y2, z2 = (g(a, k) for k in range(3) for a in (xn, yn, zn))
    eps = _c(K_EPSILON, verts)
    zmax = torch.fmax(torch.fmax(z0, z1), z2)
    ok = ~(zmax < 0) & ~(_edge(x0, y0, x1, y1, x2, y2).abs() <= eps)
    # NDC x decreases with the column, y with the row: index i = W-1-xi (H-1-yi) increases with x (y)
    xmin, xmax = torch.fmin(torch.fmin(x0, x1), x2), torch.fmax(torch.fmax(x0, x1), x2)
    ymin, ymax = torch.fmin(torch.fmin(y0, y1), y2), torch.fmax(torch.fmax(y0, y1), y2)
    ix0, ix1 = _pixel_range(xmin, xmax, W, H)
    iy0, iy1 = _pixel_range(ymin, ymax, H, W)
    nx, ny = (ix1 - ix0 + 1) * ok, (iy1 - iy0 + 1) * ok
    cnt = (nx * ny).reshape(-1)
    sel = torch.repeat_interleave(torch.arange(B * F, device=dev), cnt)     # one entry per (face, box pixel)
    start = torch.cumsum(cnt, 0) - cnt
    k = torch.arange(sel.numel(), device=dev) - start[sel]
    nxs = nx.reshape(-1)[sel]
    ix = ix0.reshape(-1)[sel] + k % nxs
    iy = iy0.reshape(-1)[sel] + k // nxs
    b, f = sel // F, sel % F
    px, py = pix_to_ndc(ix, W, H, verts), pix_to_ndc(iy, H, W, verts)
    fl = lambda a: a.reshape(-1)[sel]
    cov, w0, w1, w2, pz = pixel_test(px, py, *(fl(a) for a in (x0, y0, z0, x1, y1, z1, x2, y2, z2)))
    pix = (b * H + (H - 1 - iy)) * W + (W - 1 - ix)                          # flat [B,H,W] index of (yi, xi)
    pix, f, pz = pix[cov], f[cov], pz[cov]
    n = B * H * W
    best = torch.full((n,), torch.iinfo(torch.int64).max, dtype=torch.int64, device=dev)
    if dtype == torch.float32:
        best.scatter_reduce_(0, pix, depth_key(pz, f), "amin")
        hit = best != torch.iinfo(torch.int64).max
        face = torch.where(hit, best & 0xFFFFFFFF, torch.full_like(best, -1))
    else:
        zmin = torch.full((n,), math.inf, dtype=dtype, device=dev).scatter_reduce_(0, pix, pz, "amin")
        at = pz == zmin[pix]
        best.scatter_reduce_(0, pix[at], f[at], "amin")
        hit = best != torch.iinfo(torch.int64).max
        face = torch.where(hit, best, torch.full_like(best, -1))
    # resolve: recompute the winner's barycentrics at each covered pixel with the same arithmetic
    q = hit.nonzero().squeeze(1)
    qb, qf = q // (H * W), face[q]
    yi, xi = (q // W) % H, q % W
    px, py = pix_to_ndc(W - 1 - xi, W, H, verts), pix_to_ndc(H - 1 - yi, H, W, verts)
    at = lambda a: a[qb, qf]
    _, w0, w1, w2, pz = pixel_test(px, py, *(at(a) for a in (x0, y0, z0, x1, y1, z1, x2, y2, z2)))
    zbuf = torch.full((n,), -1.0, dtype=dtype, device=dev)
    bary = torch.full((n, 3), -1.0, dtype=dtype, device=dev)
    zbuf[q] = pz
    bary[q] = torch.stack([w0, w1, w2], -1)
    return face.reshape(B, H, W), zbuf.reshape(B, H, W), bary.reshape(B, H, W, 3)


# ---- stand-ins with pytorch3d's call shapes (what lib/data/preprocessor.py:9-10 imports) ------------------------------------
Fragments = namedtuple("Fragments", "pix_to_face zbuf bary_coords dists")


class Meshes:
    """pytorch3d.structures.Meshes for a batch of equal-sized meshes (verts [B,V,3], faces [B,F,3])."""

    def __init__(self, verts, faces):
        self._verts, self._faces = torch.as_tensor(verts), torch.as_tensor(faces)

    def to(self, device):
        return Meshes(self._verts.to(device), self._faces.to(device))

    def verts_padded(self):
        return self._verts

    def faces_padded(self):
        return self._faces


class PerspectiveCameras:
    def __init__(self, focal_length=1.0, R=None, T=None, in_ndc=True, device="cpu", principal_point=None, **kwargs):
        if not in_ndc or principal_point is not None or kwargs:
            raise RuntimeError("PerspectiveCameras stand-in: only in_ndc=True with principal point 0")
        focal = torch.as_tensor(focal_length, dtype=torch.float32)
        if focal.numel() != 1:
            raise RuntimeError("PerspectiveCameras stand-in: one focal length shared by the batch")
        self.focal, self.R, self.T = float(focal.reshape(())), R.to(device), T.to(device)


class RasterizationSettings:
    def __init__(self, image_size=256, blur_radius=0.0, faces_per_pixel=1, cull_backfaces=False, perspective_correct=None,
                 **kwargs):
        if blur_radius != 0.0 or faces_per_pixel != 1 or cull_backfaces or perspective_correct is False:
            raise RuntimeError("RasterizationSettings stand-in: blur_radius 0, faces_per_pixel 1, no culling, perspective-correct")
        self.image_size = (image_size, image_size) if isinstance(image_size, int) else tuple(image_size)


class MeshRasterizer:
    def __init__(self, cameras=None, raster_settings=None):
        self.cameras, self.raster_settings = cameras, raster_settings

    def __call__(self, meshes, cameras=None, dtype=torch.float32):
        """-> Fragments(pix_to_face [B,H,W,1] PACKED (b * F + face, -1 background), zbuf [B,H,W,1], bary [B,H,W,1,3],
        dists [B,H,W,1]).  dists is not restated (-1 everywhere): the reference discards it."""
        cams = cameras or self.cameras
        H, W = self.raster_settings.image_size
        verts, faces = meshes.verts_padded(), meshes.faces_padded()
        if not bool((faces == faces[:1]).all()):
            raise RuntimeError("MeshRasterizer stand-in: the meshes of a batch share one face list")
        p2f, zbuf, bary = rasterize(verts, faces[0], cams.R, cams.T, cams.focal, H, W, dtype=dtype)
        F = faces.shape[1]
        off = torch.arange(verts.shape[0], device=p2f.device)[:, None, None] * F
        p2f = torch.where(p2f >= 0, p2f + off, p2f)
        return Fragments(p2f[..., None], zbuf[..., None], bary[..., None, :], torch.full_like(zbuf[..., None], -1.0))


# ---- the oracle preprocessor: lib/data/preprocessor.py:14-176 with the stand-ins, device-aware ------------------------------
class SHHQPreprocessor(torch.nn.Module):
    def __init__(self, gen_height, gen_width, **kwargs):
        super().__init__()
        self.height, self.width = gen_height, gen_width
        self.mode = kwargs.get("coordinate_mode", "fix_body")
        if self.mode != "fix_body":
            raise RuntimeError("oracle SHHQPreprocessor: only coordinate_mode='fix_body'")
        self.register_buffer("vertex_approximation", torch.zeros([6890], dtype=torch.long))
        self.register_buffer("smpl_faces", torch.zeros([13776, 3], dtype=torch.long))
        self.register_buffer("smpl_faces_to_labels", torch.zeros([13776], dtype=torch.long))
        self.rasterizer = MeshRasterizer(raster_settings=RasterizationSettings(image_size=(gen_height, gen_width)))

    @torch.no_grad()
    def init_smpl(self, smpl_faces, smpl_faces_to_labels):
        self.smpl_faces.copy_(smpl_faces)
        self.smpl_faces_to_labels.copy_(smpl_faces_to_labels)

    @torch.no_grad()
    def forward(self, data, rotate=False, **kwargs):
        B = data["scales"].shape[0]
        h = torch.randn(B) * (kwargs["h_stddev"] if rotate else 0) + kwargs["h_mean"]
        v = torch.randn(B) * (kwargs["v_stddev"] if rotate else 0) + kwargs["v_mean"]
        return self.forward_with_rotation(data, h, v, torch.zeros_like(h), **kwargs)

    @torch.no_grad()
    def forward_with_rotation(self, data, h_rotation, v_rotation, r_rotation, dtype=torch.float32, **kwargs):
        dev = data["scales"].device
        B = data["scales"].shape[0]
        euler = torch.zeros([B, 3], device=dev)
        euler[:, 1] = -h_rotation
        euler[:, 0] = math.pi - v_rotation
        euler[:, 2] = -r_rotation
        R = data["full_pose"][:, 0] @ euler_xyz_to_matrix(euler)
        R_raster = torch.inverse(R)
        body = torch.nn.functional.pad(R, (0, 1, 0, 1), mode="constant", value=0.0)
        body[:, -1, -1] = 1.0
        data["cam2world_matrices"] = torch.inverse(torch.bmm(torch.bmm(data["R"], data["T"]), body).float())

        faces = self.smpl_faces.unsqueeze(0).repeat(B, 1, 1)
        meshes = Meshes(verts=data["vertices"], faces=faces).to(dev)
        focal_raster = 1.0 / math.tan(math.pi * 1 / 180 / 2)
        T_raster = data["T"][:, :3, -1].clone()
        T_raster[:, -1] = focal_raster / data["scales"] * 0.5
        cameras = PerspectiveCameras(focal_length=-focal_raster, R=R_raster, T=T_raster, in_ndc=True, device=dev)
        pix_to_face, zbuf, bary, _ = self.rasterizer(meshes, cameras=cameras, dtype=dtype)
        pix_to_face = pix_to_face.reshape(B, self.height, self.width)
        bg = pix_to_face < 0
        pix_to_face = pix_to_face % len(self.smpl_faces)
        self.last_pix_to_face = torch.where(bg, -1, pix_to_face)          # kept for the tests: per-mesh face, -1 background
        pix_to_face_verts = self.smpl_faces[pix_to_face]
        pix_to_vert = torch.gather(pix_to_face_verts, dim=-1, index=torch.argmax(bary[:, :, :, 0, :], dim=-1, keepdim=True))
        pix_to_vert = pix_to_vert.reshape(B, self.height, self.width)
        pix_to_vert[bg] = -1
        sem = data["tpose_vertices"][0][pix_to_vert]
        sem[bg.unsqueeze(-1).expand_as(sem)] = 0
        data["rasterized_semantics"] = sem.permute(0, 3, 1, 2)
        seg = self.smpl_faces_to_labels[pix_to_face] + 2
        seg[bg] = 1
        data["rasterized_segments"] = seg
        return data
