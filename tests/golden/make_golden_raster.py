"""Fixture for the preprocessor's rasterisation step (SURVEY.md 8f-2) from the reference's OWN code (build container only).

The data dict is built from `synthetic.make_body_mesh` (a closed body-like surface with SMPL's 6 890 vertices / 13 776 faces;
SMPL_NEUTRAL.pkl and densepose_data.json are licence-gated and absent) posed with seeded betas / pose / camera through
oracle/smpl_port.py in float64 (so that the fp32 inputs are reproducible bit for bit), the way make_golden_smpl.py does.  Then
the reference's `SHHQPreprocessor.__init__ / init_smpl / forward_with_rotation` (lib/data/preprocessor.py:14-176, hence
`_forward_fix_body` + `_forward_rasterize`) run unmodified, with pytorch3d's `PerspectiveCameras / MeshRasterizer /
RasterizationSettings / Meshes / euler_angles_to_matrix` supplied by oracle/raster_port.py and oracle/smpl_port.py.
Cases: B = 3 at 256x128 (MAP3DBN) and B = 2 at 512x256 (MAP3DBN512 / 512L); rotations drawn at the curricula's
h_stddev = 0.4, v_stddev = 0.1.

Writes tests/golden/raster_pins.npz: per case `c<i>_cam2world`, `c<i>_pix_to_face` (int16, per-mesh face, -1 background, as
the rasteriser returned it to the reference's code), `c<i>_segments` (uint8), and `rasterized_semantics` in full for case 0,
as every 7th element + the float64 norm of the whole tensor for case 1.  tests/test_cpu_raster_pin.py re-creates the inputs
with `inputs()`."""
import importlib
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CASES = [dict(B=3, H=256, W=128, seed=21), dict(B=2, H=512, W=256, seed=22)]
SEM_STRIDE = 7


def inputs(case):
    """-> (faces [F,3] int64, faces_to_labels [F] int64, data dict (fp32, CPU), h, v, r rotations [B])."""
    from oracle import smpl_port as sp
    syn = importlib.import_module("3dhumangan_b200.synthetic")
    mesh = syn.make_body_mesh(seed=0)
    m = {k: (v.double() if v.is_floating_point() else v) for k, v in mesh["smpl"].items()}
    B = case["B"]
    g = torch.Generator().manual_seed(case["seed"])
    betas = torch.randn(B, 10, generator=g, dtype=torch.float64) * 0.5
    pose = torch.randn(B, 24, 3, generator=g, dtype=torch.float64) * 0.3
    orig_cam = torch.stack([1.2 + 0.2 * torch.rand(B, generator=g, dtype=torch.float64), torch.ones(B, dtype=torch.float64),
                            0.1 * torch.randn(B, generator=g, dtype=torch.float64), 0.1 * torch.randn(B, generator=g, dtype=torch.float64)], 1)
    h = (torch.randn(B, generator=g) * 0.4).float()
    v = (torch.randn(B, generator=g) * 0.1).float()
    A, v_shaped, _, _, Jt = sp.lbs(betas, pose.reshape(B, -1), m["v_template"], m["shapedirs"], m["posedirs"], m["J_regressor"],
                                   m["parents"], m["lbs_weights"])
    rot = sp.batch_rodrigues(pose.reshape(-1, 3)).reshape(B, 24, 3, 3)
    cond = sp.conditions_fix_body(orig_cam, Jt, rot, v_shaped, A, m["lbs_weights"], m["v_template"])
    cond = {k: v_.float().contiguous() for k, v_ in cond.items()}
    return mesh["faces"], mesh["faces_to_labels"], cond, h, v, torch.zeros(B)


def main():
    sys.path.insert(0, os.path.join(ROOT, "oracle", "shims"))
    sys.path.insert(0, os.environ["HG_REFERENCE"])           # a checkout of the reference
    from oracle import raster_port as rp
    from oracle import smpl_port as sp
    import lib.data.preprocessor as pp
    for n in ("PerspectiveCameras", "MeshRasterizer", "RasterizationSettings", "Meshes"):
        setattr(pp, n, getattr(rp, n))
    pp.euler_angles_to_matrix = lambda e, convention: sp.euler_xyz_to_matrix(e)
    seen = []
    call = rp.MeshRasterizer.__call__
    rp.MeshRasterizer.__call__ = lambda self, *a, **k: seen.append(call(self, *a, **k)) or seen[-1]
    out = {}
    for i, case in enumerate(CASES):
        faces, labels, cond, h, v, r = inputs(case)
        pre = pp.SHHQPreprocessor(gen_height=case["H"], gen_width=case["W"])
        pre.init_smpl(faces, labels)
        data = pre.forward_with_rotation(dict(cond), h, v, r)
        B, H, W = case["B"], case["H"], case["W"]
        p2f = seen[-1].pix_to_face.reshape(B, H, W)
        p2f = torch.where(p2f >= 0, p2f % faces.shape[0], p2f)
        sem = data["rasterized_semantics"]
        out[f"c{i}_cam2world"] = data["cam2world_matrices"].numpy()
        out[f"c{i}_pix_to_face"] = p2f.numpy().astype(np.int16)
        out[f"c{i}_segments"] = data["rasterized_segments"].numpy().astype(np.uint8)
        if i == 0:
            out[f"c{i}_semantics"] = sem.contiguous().numpy()
        else:
            out[f"c{i}_semantics_sample"] = sem.reshape(-1)[::SEM_STRIDE].numpy()
            out[f"c{i}_semantics_norm"] = np.array(float(sem.double().norm()))
        print(f"case {i}: B={B} {H}x{W}, body pixels {int((p2f >= 0).sum())}, labels {sorted(set(data['rasterized_segments'].unique().tolist()))}")
    np.savez_compressed(os.path.join(HERE, "raster_pins.npz"), **out)


if __name__ == "__main__":
    main()
