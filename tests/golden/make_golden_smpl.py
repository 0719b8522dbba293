"""Fixture for the SMPL condition step (SURVEY.md 8f-4) from the reference's OWN code (build container only).

Runs, on seeded synthetic SMPL-like data (SMPL_NEUTRAL.pkl is licence-gated and absent):
  * `lib.components.smpl.lbs` (the reference's function body) with the four smplx.lbs helpers it imports supplied by
    oracle/smpl_port.py (smplx itself is not installed);
  * `SHHQDataset._preprocess_smpl_fix_body` (unbound, on a stand-in `self`) per sample;
  * `SHHQPreprocessor._forward_fix_body` (unbound) with pytorch3d's `euler_angles_to_matrix` supplied by the oracle.
Writes tests/golden/smpl_conditions.npz (inputs are re-created from the seeds by tests/test_oracle_pin.py)."""
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle", "shims"))


def inputs(seed=0, B=3, V=500, J=24, NB=10):
    g = torch.Generator().manual_seed(seed)
    parents = torch.tensor([-1] + [max(0, (i - 1) // 2) for i in range(1, J)], dtype=torch.int64)
    model = dict(v_template=(torch.rand(V, 3, generator=g) - 0.5) * torch.tensor([0.9, 1.7, 0.3]), shapedirs=torch.randn(V, 3, NB, generator=g) * 0.01,
                 posedirs=torch.randn((J - 1) * 9, V * 3, generator=g) * 0.01, J_regressor=torch.softmax(torch.randn(J, V, generator=g) * 3, 1),
                 parents=parents, lbs_weights=torch.softmax(torch.randn(V, J, generator=g) * 4, 1))
    betas = torch.randn(B, NB, generator=g)
    pose = torch.randn(B, J, 3, generator=g) * 0.4
    orig_cam = torch.stack([1.2 + 0.2 * torch.rand(B, generator=g), 1.2 + 0.2 * torch.rand(B, generator=g),
                            0.1 * torch.randn(B, generator=g), 0.1 * torch.randn(B, generator=g)], 1)
    angles = torch.randn(3, B, generator=g) * 0.3
    return model, betas, pose, orig_cam, angles


def main():
    sys.path.insert(0, os.environ["HG_REFERENCE"])           # a checkout of the reference
    from oracle import smpl_port as sp
    import lib.components.smpl as rsmpl
    for n in ("blend_shapes", "vertices2joints", "batch_rodrigues", "batch_rigid_transform"):
        setattr(rsmpl, n, getattr(sp, n))
    model, betas, pose, orig_cam, angles = inputs()
    A, v_shaped, verts, J, Jt = rsmpl.lbs(betas, pose.reshape(betas.shape[0], -1), model["v_template"], model["shapedirs"], model["posedirs"],
                                          model["J_regressor"], model["parents"], model["lbs_weights"])
    rot = sp.batch_rodrigues(pose.reshape(-1, 3)).reshape(betas.shape[0], -1, 3, 3)
    import lib.data.datasets as ds
    import lib.data.preprocessor as pp
    pp.euler_angles_to_matrix = lambda e, convention: sp.euler_xyz_to_matrix(e)
    fake = types.SimpleNamespace(joints=list(range(24)), smpl_tpose_vertices=model["v_template"].numpy().copy(), inference=False)
    outs = []
    for b in range(betas.shape[0]):
        pred = {"orig_cam": orig_cam[b:b + 1].numpy(), "joints": Jt[b:b + 1].numpy(), "full_pose": rot[b:b + 1].numpy(),
                "tpose_vertices": v_shaped[b:b + 1].numpy(), "fk_matrices": A[b:b + 1].numpy(), "lbs_weights": model["lbs_weights"].numpy()}
        outs.append(ds.SHHQDataset._preprocess_smpl_fix_body(fake, pred))
    cond = {k: torch.from_numpy(np.stack([np.asarray(o[k], dtype=np.float32) for o in outs])) for k in outs[0]}
    fake_p = types.SimpleNamespace(device="cpu")
    data, R_raster = pp.SHHQPreprocessor._forward_fix_body.__wrapped__(fake_p, dict(cond), angles[0], angles[1], angles[2]) \
        if hasattr(pp.SHHQPreprocessor._forward_fix_body, "__wrapped__") else pp.SHHQPreprocessor._forward_fix_body(fake_p, dict(cond), angles[0], angles[1], angles[2])
    np.savez_compressed(os.path.join(HERE, "smpl_conditions.npz"), A=A.numpy(), v_shaped=v_shaped.numpy(), verts=verts.numpy(), J=J.numpy(),
                        Jt=Jt.numpy(), cam2world=data["cam2world_matrices"].numpy(), R_raster=R_raster.numpy(),
                        **{"cond_" + k: v.numpy() for k, v in cond.items()})
    print("written", {k: tuple(v.shape) for k, v in cond.items()})


if __name__ == "__main__":
    main()
