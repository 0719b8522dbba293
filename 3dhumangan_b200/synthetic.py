"""Procedural SMPL-like `conditions` for benchmarks, tests and smoke runs.

The reference feeds `Map3DGenerator.forward/render` with a `conditions` dict built by
`SHHQDataset._preprocess_smpl_fix_body` (lib/data/datasets.py:117-181) and
`SHHQPreprocessor._forward_fix_body` (lib/data/preprocessor.py:72-98) from SMPL fits of real
photographs.  `SMPL_NEUTRAL.pkl` is licence-gated and absent, so this module synthesises
tensors with the same keys, shapes, dtypes and value ranges (SURVEY.md §8d):

    skeletons_xyz [B,24,3]   vertices [B,6890,3]   tpose_vertices [B,6890,3]
    fk_matrices [B,24,4,4]   lbs_weights [B,6890,24]   cam2world_matrices [B,4,4]
    intrinsics [B,4,4]       scales [B]

A 24-joint kinematic tree (SMPL topology) is posed with per-joint axis-angle noise, 6890
vertices are scattered on capsules around the bones and skinned with the same linear-blend
formula as datasets.py:152-155.  Everything is generated on the CPU from a seeded
`torch.Generator`, so the same seed gives bit-identical inputs to the oracle and the kernels.
"""
from __future__ import annotations

import math

import torch

N_JOINTS = 24
N_VERTS = 6890

# SMPL kinematic tree (parent of joint j); joint 0 = pelvis.
_PARENTS = [-1, 0, 0, 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 9, 9, 12, 13, 14, 16, 17, 18, 19, 20, 21]

# Rest-pose joint positions (metres, y up, roughly SMPL's neutral T-pose).
_REST = [
    (0.00, -0.24, 0.03), (0.06, -0.33, 0.02), (-0.06, -0.33, 0.02), (0.00, -0.12, 0.00),
    (0.10, -0.71, 0.02), (-0.10, -0.71, 0.02), (0.00, 0.02, 0.01), (0.09, -1.11, -0.02),
    (-0.09, -1.11, -0.02), (0.00, 0.07, 0.03), (0.11, -1.17, 0.10), (-0.11, -1.17, 0.10),
    (0.00, 0.28, -0.01), (0.08, 0.19, 0.00), (-0.08, 0.19, 0.00), (0.00, 0.37, 0.04),
    (0.17, 0.23, -0.01), (-0.17, 0.23, -0.01), (0.43, 0.22, -0.03), (-0.43, 0.22, -0.03),
    (0.68, 0.22, -0.03), (-0.68, 0.22, -0.03), (0.77, 0.21, -0.04), (-0.77, 0.21, -0.04),
]


def _rodrigues(aa: torch.Tensor) -> torch.Tensor:
    """axis-angle [...,3] -> rotation matrices [...,3,3] (float64)."""
    theta = aa.norm(dim=-1, keepdim=True).clamp_min(1e-12)
    k = aa / theta
    K = torch.zeros(aa.shape[:-1] + (3, 3), dtype=aa.dtype)
    K[..., 0, 1], K[..., 0, 2] = -k[..., 2], k[..., 1]
    K[..., 1, 0], K[..., 1, 2] = k[..., 2], -k[..., 0]
    K[..., 2, 0], K[..., 2, 1] = -k[..., 1], k[..., 0]
    s = torch.sin(theta)[..., None]
    c = torch.cos(theta)[..., None]
    eye = torch.eye(3, dtype=aa.dtype).expand_as(K)
    return eye + s * K + (1 - c) * (K @ K)


def make_template(gen: torch.Generator):
    """Template mesh: vertices on capsules around bones + <=4-sparse LBS weights (rows sum to 1)."""
    rest = torch.tensor(_REST, dtype=torch.float64)
    bones = [(j, p) for j, p in enumerate(_PARENTS) if p >= 0]
    nb = len(bones)
    which = torch.randint(0, nb, (N_VERTS,), generator=gen)
    t = torch.rand(N_VERTS, generator=gen, dtype=torch.float64)
    ang = torch.rand(N_VERTS, generator=gen, dtype=torch.float64) * 2 * math.pi
    rad = 0.03 + 0.06 * torch.rand(N_VERTS, generator=gen, dtype=torch.float64)
    a = torch.stack([rest[j] for j, _ in bones])[which]
    b = torch.stack([rest[p] for _, p in bones])[which]
    axis = b - a
    axis = axis / axis.norm(dim=-1, keepdim=True).clamp_min(1e-9)
    helper = torch.tensor([0.0, 0.0, 1.0], dtype=torch.float64).expand_as(axis).clone()
    near_z = axis[:, 2].abs() > 0.9
    helper[near_z] = torch.tensor([1.0, 0.0, 0.0], dtype=torch.float64)
    u = torch.linalg.cross(axis, helper)
    u = u / u.norm(dim=-1, keepdim=True)
    v = torch.linalg.cross(axis, u)
    verts = a + (b - a) * t[:, None] + rad[:, None] * (torch.cos(ang)[:, None] * u + torch.sin(ang)[:, None] * v)
    # distance-softmax skinning weights, keep the 4 nearest joints
    d = torch.cdist(verts, rest)
    w = torch.softmax(-d / 0.05, dim=-1)
    top = torch.topk(w, 4, dim=-1)
    lbs = torch.zeros_like(w).scatter_(1, top.indices, top.values)
    lbs = lbs / lbs.sum(-1, keepdim=True)
    return rest, verts, lbs


def make_conditions(batch_size: int, seed: int = 1, pose_std: float = 0.3, view_std: float = 0.4,
                    scale: float = 0.7, device="cpu", canonical_pose: bool = False):
    """Build the `conditions` dict (float32) for `batch_size` bodies."""
    gen = torch.Generator().manual_seed(seed)
    rest, tverts, lbs = make_template(gen)
    B = batch_size
    fov = math.pi * 12 / 180                      # datasets.py:119-120
    focal = 1.0 / math.tan(fov / 2)

    aa = torch.randn(B, N_JOINTS, 3, generator=gen, dtype=torch.float64) * (0.0 if canonical_pose else pose_std)
    R = _rodrigues(aa)
    G = torch.zeros(B, N_JOINTS, 4, 4, dtype=torch.float64)
    for j, p in enumerate(_PARENTS):
        L = torch.eye(4, dtype=torch.float64).repeat(B, 1, 1)
        L[:, :3, :3] = R[:, j]
        L[:, :3, 3] = rest[j] - (rest[p] if p >= 0 else 0)
        G[:, j] = L if p < 0 else G[:, p] @ L
    joints = G[:, :, :3, 3].clone()
    # rigid transforms relative to the rest pose (what SMPL calls A_j): x_posed = A_j [x_rest; 1]
    A = G.clone()
    A[:, :, :3, 3] = G[:, :, :3, 3] - torch.einsum("bjik,jk->bji", G[:, :, :3, :3], rest)
    # canonical frame: rotate pi about x (datasets.py:143-147) so the head points to -y (image top)
    cano = torch.diag(torch.tensor([1.0, -1.0, -1.0, 1.0], dtype=torch.float64))
    fk = torch.einsum("ij,bnjk->bnik", cano, A)
    vfk = torch.einsum("vj,bjkl->bvkl", lbs, fk)
    th = torch.cat([tverts, torch.ones(N_VERTS, 1, dtype=torch.float64)], -1)
    verts = torch.einsum("bvij,vj->bvi", vfk, th)[..., :3]
    skel = torch.einsum("ij,bnj->bni", cano[:3, :3], joints)
    tpose = tverts.clone()
    tpose[:, 1] += 0.35                            # datasets.py:159-160

    # camera: world2cam = R(=I) . T . body_rotation  (preprocessor.py:91-94)
    h_rot = torch.randn(B, generator=gen, dtype=torch.float64) * view_std
    w2c = torch.eye(4, dtype=torch.float64).repeat(B, 1, 1)
    c, s = torch.cos(h_rot), torch.sin(h_rot)
    w2c[:, 0, 0], w2c[:, 0, 2], w2c[:, 2, 0], w2c[:, 2, 2] = c, s, -s, c
    T = torch.eye(4, dtype=torch.float64).repeat(B, 1, 1)
    T[:, 2, 3] = focal / scale
    w2c = T @ w2c
    c2w = torch.linalg.inv(w2c)

    K = torch.eye(4, dtype=torch.float64).repeat(B, 1, 1)
    K[:, 0, 0] = focal
    K[:, 1, 1] = focal
    f32 = lambda x: x.to(torch.float32).contiguous().to(device)
    return {
        "skeletons_xyz": f32(skel),
        "vertices": f32(verts),
        "tpose_vertices": f32(tpose[None].repeat(B, 1, 1)),
        "fk_matrices": f32(fk),
        "lbs_weights": f32(lbs[None].repeat(B, 1, 1)),
        "cam2world_matrices": f32(c2w),
        "intrinsics": f32(K),
        "scales": f32(torch.full((B,), scale, dtype=torch.float64)),
    }


def make_body_mesh(seed: int = 0):
    """A closed genus-0 body-like surface with SMPL's counts, for the preprocessor's rasteriser (`raster.py`).

    A UV sphere of 82 rings x 84 segments + 2 poles has exactly V = 6 890 vertices and F = 13 776 faces.  It is stretched to a
    body's proportions (y up, head at +y, like SMPL's template) and its radius is modulated by seeded waves and signed Gaussian
    bumps, so the surface is not convex and a rotated view has real self-occlusions.  Faces are labelled over 24 classes by
    height band (12) x side (2) of their centroid, standing in for `densepose_data.json`'s face labels.

    -> dict(vertices [V,3] float32, faces [F,3] int64, faces_to_labels [F] int64, smpl=dict(v_template, shapedirs [V,3,10],
    posedirs [207, V*3], J_regressor [24,V], parents [24], lbs_weights [V,24])); `smpl.SMPLModel.from_arrays(**mesh["smpl"])`
    skins it with smooth blend shapes and distance-based weights around `_REST`'s joints.  Pure CPU torch, seeded."""
    gen = torch.Generator().manual_seed(seed)
    rings, segs = 82, 84
    theta = math.pi * torch.arange(1, rings + 1, dtype=torch.float64) / (rings + 1)
    phi = 2 * math.pi * torch.arange(segs, dtype=torch.float64) / segs
    th, ph = theta[:, None].expand(rings, segs).reshape(-1), phi[None].expand(rings, segs).reshape(-1)
    th = torch.cat([torch.zeros(1, dtype=torch.float64), th, torch.full((1,), math.pi, dtype=torch.float64)])
    ph = torch.cat([torch.zeros(1, dtype=torch.float64), ph, torch.zeros(1, dtype=torch.float64)])
    n = torch.stack([torch.sin(th) * torch.cos(ph), torch.cos(th), torch.sin(th) * torch.sin(ph)], -1)
    p = torch.rand(4, generator=gen, dtype=torch.float64) * 2 * math.pi
    r = 1.0 + 0.15 * torch.sin(3 * ph + p[0]) * torch.sin(2 * th) + 0.1 * torch.cos(5 * th + p[1]) \
        + 0.06 * torch.sin(7 * ph + p[2]) * torch.sin(th) ** 2
    centres = torch.nn.functional.normalize(torch.randn(14, 3, generator=gen, dtype=torch.float64), dim=-1)
    amp = (torch.rand(14, generator=gen, dtype=torch.float64) - 0.4) * 0.7            # mostly outward bumps, some dents
    r = r + (amp * torch.exp(-(1 - n @ centres.T) / 0.02)).sum(-1)
    verts = n * r[:, None] * torch.tensor([0.32, 0.85, 0.17], dtype=torch.float64) + torch.tensor([0.0, -0.4, 0.0], dtype=torch.float64)

    V = 2 + rings * segs
    ring = lambda k, j: 1 + k * segs + j % segs
    j = torch.arange(segs)
    faces = [torch.stack([torch.zeros_like(j), ring(0, j), ring(0, j + 1)], -1)]
    for k in range(rings - 1):
        a, b, c, d = ring(k, j), ring(k, j + 1), ring(k + 1, j), ring(k + 1, j + 1)
        faces += [torch.stack([a, c, b], -1), torch.stack([b, c, d], -1)]
    faces.append(torch.stack([torch.full_like(j, V - 1), ring(rings - 1, j + 1), ring(rings - 1, j)], -1))
    faces = torch.cat(faces).to(torch.int64)
    cen = verts[faces].mean(1)
    y0, y1 = verts[:, 1].min(), verts[:, 1].max()
    band = ((cen[:, 1] - y0) / (y1 - y0) * 12).floor().clamp(0, 11).to(torch.int64)
    labels = band * 2 + (cen[:, 0] > 0).to(torch.int64)

    rest = torch.tensor(_REST, dtype=torch.float64)
    d = torch.cdist(verts, rest)
    w = torch.softmax(-d / 0.08, dim=-1)
    top = torch.topk(w, 4, dim=-1)
    lbs = torch.zeros_like(w).scatter_(1, top.indices, top.values)
    lbs = lbs / lbs.sum(-1, keepdim=True)
    jreg = torch.softmax(-d.T / 0.05, dim=-1)
    wave = lambda k: torch.sin(verts @ (torch.randn(3, k, generator=gen, dtype=torch.float64) * 3)
                               + torch.rand(k, generator=gen, dtype=torch.float64) * 2 * math.pi)
    shapedirs = 0.02 * wave(30).reshape(V, 10, 3).transpose(1, 2)
    posedirs = 0.003 * wave(207 * 3).reshape(V, 207, 3).permute(1, 0, 2).reshape(207, V * 3)
    f32 = lambda t: t.to(torch.float32).contiguous()
    return {"vertices": f32(verts), "faces": faces, "faces_to_labels": labels,
            "smpl": dict(v_template=f32(verts), shapedirs=f32(shapedirs), posedirs=f32(posedirs), J_regressor=f32(jreg),
                         parents=torch.tensor(_PARENTS, dtype=torch.int64), lbs_weights=f32(lbs))}
