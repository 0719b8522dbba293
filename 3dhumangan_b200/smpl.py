"""SMPL skinning and the generator's pose conditions on the device (SURVEY.md 8f-4) -- the step in front of the hot path that the
reference runs on the CPU per sample: `lbs` (lib/components/smpl.py:11-107, built on smplx.lbs),
`SHHQDataset._preprocess_smpl_fix_body` (lib/data/datasets.py:117-181) and the view rotation of
`SHHQPreprocessor._forward_fix_body` (lib/data/preprocessor.py:72-98).  With a real `SMPL_NEUTRAL.pkl` (licence-gated, not in
this image) `SMPLModel.from_arrays` takes its arrays; tests and benchmarks use `SMPLModel.synthetic`.

    model = SMPLModel.synthetic(device)                       # or .from_arrays(v_template, shapedirs, posedirs, J_regressor, parents, lbs_weights)
    out   = lbs(betas [B,10], pose [B,24,3], model)           # fk_matrices (A), tpose_vertices (v_shaped), vertices, joints
    cond  = conditions_fix_body(orig_cam [B,4], out, model)   # the dict Map3DGenerator.forward reads (+ R, T, cano_matrices, full_pose)
    cond["cam2world_matrices"] = cam2world_fix_body(cond, h, v, r)

Skinning runs on csrc/smpl.cu (`hg_smpl_shape`, `hg_smpl_pose`, `hg_smpl_skin`); the handful of 4x4 products around it are
batched torch calls.  No gradients (the reference treats the conditions as data)."""
from __future__ import annotations

import math
from dataclasses import dataclass

import torch
import torch.nn.functional as F

from . import abi


@dataclass
class SMPLModel:
    v_template: torch.Tensor      # [V,3]
    shapedirs: torch.Tensor       # [V,3,NB]
    posedirs: torch.Tensor        # [(J-1)*9, V*3]
    J_regressor: torch.Tensor     # [J,V]
    parents: torch.Tensor         # [J] int32, parents[0] = -1
    lbs_weights: torch.Tensor     # [V,J]

    @staticmethod
    def from_arrays(v_template, shapedirs, posedirs, J_regressor, parents, lbs_weights, device="cuda"):
        f = lambda t: torch.as_tensor(t, dtype=torch.float32).to(device).contiguous()
        return SMPLModel(f(v_template), f(shapedirs), f(posedirs), f(J_regressor),
                         torch.as_tensor(parents, dtype=torch.int32).to(device).contiguous(), f(lbs_weights))

    @staticmethod
    def synthetic(device="cuda", V=6890, J=24, NB=10, seed=0):
        """A structurally valid stand-in (kinematic tree, sparse convex skinning weights, small blend shapes)."""
        g = torch.Generator().manual_seed(seed)
        parents = torch.tensor([-1] + [max(0, (i - 1) // 2) for i in range(1, J)], dtype=torch.int32)
        v = (torch.rand(V, 3, generator=g) - 0.5) * torch.tensor([0.9, 1.7, 0.3])
        w = torch.rand(V, J, generator=g) ** 8
        top = torch.topk(w, 4, dim=1)
        w = torch.zeros(V, J).scatter_(1, top.indices, top.values)
        w = w / w.sum(1, keepdim=True)
        jr = torch.rand(J, V, generator=g) ** 20
        jr = jr / jr.sum(1, keepdim=True)
        return SMPLModel.from_arrays(v, torch.randn(V, 3, NB, generator=g) * 0.01, torch.randn((J - 1) * 9, V * 3, generator=g) * 0.01,
                                     jr, parents, w, device)


@torch.no_grad()
def lbs(betas, pose, model: SMPLModel, pose2rot=True):
    """-> dict(fk_matrices [B,J,4,4] (the rigid transforms A), tpose_vertices [B,V,3] (shaped), vertices [B,V,3], joints_shaped,
    joints [B,J,3] (posed), rot_mats [B,J,3,3])  --  lib/components/smpl.py:11-107 / SMPL.forward :171-205."""
    abi.require_device()
    dev = model.v_template.device
    B = betas.shape[0]
    V, J, NB = model.v_template.shape[0], model.J_regressor.shape[0], model.shapedirs.shape[2]
    betas = betas.to(dev).float().contiguous()
    pose = pose.to(dev).float().reshape(B, J, -1).contiguous()
    if pose.shape[-1] != (3 if pose2rot else 9):
        raise RuntimeError("hg3d: pose must be [B,J,3] axis-angle (pose2rot=True) or [B,J,3,3] rotation matrices")
    f32 = dict(dtype=torch.float32, device=dev)
    nblk = int(abi.lib().hg_smpl_shape_blocks(V))
    v_shaped = torch.empty(B, V, 3, **f32)
    jpart = torch.empty(B, nblk, J, 3, **f32)
    joints = torch.empty(B, J, 3, **f32)
    rot = torch.empty(B, J, 9, **f32)
    feat = torch.empty(B, (J - 1) * 9, **f32)
    A = torch.empty(B, J, 16, **f32)
    jt = torch.empty(B, J, 3, **f32)
    verts = torch.empty(B, V, 3, **f32)
    with torch.cuda.device_of(v_shaped):
        abi.call("hg_smpl_shape", abi.ptr(model.v_template), abi.ptr(model.shapedirs), abi.ptr(betas), abi.ptr(model.J_regressor),
                 abi.ptr(v_shaped), abi.ptr(jpart), B, V, NB, J, abi.stream())
        abi.call("hg_smpl_pose", abi.ptr(jpart), nblk, abi.ptr(pose), int(not pose2rot), abi.ptr(model.parents), abi.ptr(joints), abi.ptr(rot),
                 abi.ptr(feat), abi.ptr(A), abi.ptr(jt), B, J, abi.stream())
        abi.call("hg_smpl_skin", abi.ptr(v_shaped), V * 3, abi.ptr(feat), abi.ptr(model.posedirs), (J - 1) * 9, abi.ptr(model.lbs_weights), 0,
                 abi.ptr(A), abi.ptr(verts), B, V, J, abi.stream())
    return {"fk_matrices": A.reshape(B, J, 4, 4), "tpose_vertices": v_shaped, "vertices": verts, "joints_shaped": joints, "joints": jt,
            "rot_mats": rot.reshape(B, J, 3, 3), "lbs_weights": model.lbs_weights}


@torch.no_grad()
def conditions_fix_body(orig_cam, pred, model: SMPLModel, joint_ids=tuple(range(24))):
    """`SHHQDataset._preprocess_smpl_fix_body` (datasets.py:117-181) for a batch: canonicalise the body (undo the root rotation,
    flip to the y-up convention), re-skin the shaped template with the canonical transforms, camera matrices."""
    dev = model.v_template.device
    B = orig_cam.shape[0]
    V, J = model.v_template.shape[0], model.J_regressor.shape[0]
    orig_cam = orig_cam.to(dev).float()
    focal = 1.0 / math.tan(math.pi * 12 / 180 / 2)
    sx, tx, ty = orig_cam[:, 0] / 2.0, orig_cam[:, 2], orig_cam[:, 3]
    f32 = dict(dtype=torch.float32, device=dev)
    K = torch.diag(torch.tensor([focal, focal, 1.0, 1.0], **f32))[None].expand(B, 4, 4).contiguous()
    R = torch.eye(4, **f32)[None].expand(B, 4, 4).contiguous()
    T = torch.eye(4, **f32)[None].repeat(B, 1, 1)
    T[:, 0, 3], T[:, 1, 3], T[:, 2, 3] = tx, ty, focal / sx
    rot = pred["rot_mats"].double()
    cano_rot = torch.tensor([[1.0, 0.0, 0.0], [0.0, math.cos(math.pi), -math.sin(math.pi)], [0.0, math.sin(math.pi), math.cos(math.pi)]],
                            dtype=torch.float64, device=dev)
    cano = torch.eye(4, dtype=torch.float64, device=dev)[None].repeat(B, 1, 1)
    cano[:, :3, :3] = cano_rot @ torch.linalg.inv(rot[:, 0])
    fk = torch.einsum("bij,bnjk->bnik", cano, pred["fk_matrices"].double()).float().contiguous()
    verts = torch.empty(B, V, 3, **f32)
    with torch.cuda.device_of(verts):
        abi.call("hg_smpl_skin", abi.ptr(pred["tpose_vertices"].contiguous()), V * 3, None, None, 0, abi.ptr(model.lbs_weights), 0,
                 abi.ptr(fk.reshape(B, J, 16)), abi.ptr(verts), B, V, J, abi.stream())
    sk = pred["joints"][:, list(joint_ids)].double()
    sk = torch.einsum("bij,bnj->bni", cano, F.pad(sk, (0, 1), value=1.0))[..., :3].float()
    tp = model.v_template.clone()
    tp[:, 1] += 0.35
    return {"scales": sx, "skeletons_xyz": sk, "intrinsics": K, "vertices": verts, "tpose_vertices": tp[None].expand(B, V, 3).contiguous(),
            "full_pose": pred["rot_mats"], "fk_matrices": fk, "lbs_weights": model.lbs_weights[None].expand(B, V, J).contiguous(),
            "cano_matrices": cano.float(), "R": R, "T": T}


def _euler_xyz(e):
    def rot(axis, a):
        c, s, o, z = torch.cos(a), torch.sin(a), torch.ones_like(a), torch.zeros_like(a)
        m = {"X": (o, z, z, z, c, -s, z, s, c), "Y": (c, z, s, z, o, z, -s, z, c), "Z": (c, -s, z, s, c, z, z, z, o)}[axis]
        return torch.stack(m, -1).reshape(a.shape + (3, 3))
    return rot("X", e[..., 0]) @ rot("Y", e[..., 1]) @ rot("Z", e[..., 2])


@torch.no_grad()
def body_rotation(cond, h_rotation, v_rotation, r_rotation):
    """root rotation @ Euler XYZ of the view (preprocessor.py:80-87) -> [B,3,3]; its inverse is the rasteriser's R."""
    dev = cond["R"].device
    B = cond["R"].shape[0]
    euler = torch.zeros(B, 3, dtype=torch.float32, device=dev)
    euler[:, 1] = -torch.as_tensor(h_rotation, dtype=torch.float32, device=dev)
    euler[:, 0] = math.pi - torch.as_tensor(v_rotation, dtype=torch.float32, device=dev)
    euler[:, 2] = -torch.as_tensor(r_rotation, dtype=torch.float32, device=dev)
    return cond["full_pose"][:, 0] @ _euler_xyz(euler)


@torch.no_grad()
def cam2world_fix_body(cond, h_rotation, v_rotation, r_rotation, Rb=None):
    """The view rotation of `SHHQPreprocessor._forward_fix_body` (preprocessor.py:72-98) -> cam2world [B,4,4].
    `Rb`: `body_rotation(cond, h, v, r)` when the caller has it already."""
    R, T = cond["R"], cond["T"]
    if Rb is None:
        Rb = body_rotation(cond, h_rotation, v_rotation, r_rotation)
    body = F.pad(Rb, (0, 1, 0, 1))
    body[:, -1, -1] = 1.0
    return torch.inverse(torch.bmm(torch.bmm(R, T), body).float())
