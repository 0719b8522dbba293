"""The preprocessor's rasteriser (SURVEY.md 8f-2) on the CPU: the oracle (oracle/raster_port.py) against what the reference's
own `SHHQPreprocessor` code produced with it (tests/golden/raster_pins.npz, made by tests/golden/make_golden_raster.py), the
restated pytorch3d contract on hand-built cases with known answers, and the package's refusals without a device.

HAND_CASES is shared with tests/test_gpu_raster.py, which runs the same cases on the kernel."""
import importlib
import importlib.util
import os

import numpy as np
import pytest
import torch

from oracle import raster_port as rp

HERE = os.path.dirname(os.path.abspath(__file__))


def _golden_module():
    spec = importlib.util.spec_from_file_location("make_golden_raster", os.path.join(HERE, "golden", "make_golden_raster.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.parametrize("case", [0, 1])
def test_oracle_preprocessor_matches_reference_fixture(case):
    mg = _golden_module()
    gold = {k: torch.from_numpy(v) for k, v in np.load(os.path.join(HERE, "golden", "raster_pins.npz")).items()}
    c = mg.CASES[case]
    faces, labels, cond, h, v, r = mg.inputs(c)
    pre = rp.SHHQPreprocessor(gen_height=c["H"], gen_width=c["W"])
    pre.init_smpl(faces, labels)
    data = pre.forward_with_rotation(dict(cond), h, v, r)
    p = f"c{case}_"
    assert float((data["cam2world_matrices"] - gold[p + "cam2world"]).abs().max()) <= 1e-6
    p2f = pre.last_pix_to_face
    assert torch.equal(p2f, gold[p + "pix_to_face"].long())
    assert int((p2f >= 0).sum()) > 0.1 * p2f.numel()                     # the body fills a real part of the image
    seg = data["rasterized_segments"]
    assert seg.dtype == torch.int64 and seg.shape == (c["B"], c["H"], c["W"])
    assert torch.equal(seg, gold[p + "segments"].long())
    sem = data["rasterized_semantics"]
    assert sem.dtype == torch.float32 and sem.shape == (c["B"], 3, c["H"], c["W"])
    if case == 0:
        assert torch.equal(sem, gold[p + "semantics"])
    else:
        assert torch.equal(sem.reshape(-1)[::mg.SEM_STRIDE], gold[p + "semantics_sample"])
        assert abs(float(sem.double().norm()) - float(gold[p + "semantics_norm"])) <= 1e-9 * float(gold[p + "semantics_norm"])


# ---- hand-built cases: (verts [B,V,3], faces [F,3], R, T, focal, H, W) and a check on (pix_to_face, zbuf, bary) -------------
# With R = I, T = (0, 0, 1) and focal 1 a vertex (x, y, 0) projects to NDC (x, y) at depth 1.
def _flat(tris, z=None, H=8, W=8, focal=1.0, tz=1.0):
    v = torch.tensor(tris, dtype=torch.float32).reshape(1, -1, 3)
    if z is not None:
        v[0, :, 2] = torch.tensor(z, dtype=torch.float32)
    F = v.shape[1] // 3
    faces = torch.arange(3 * F).reshape(F, 3)
    return v, faces, torch.eye(3)[None], torch.tensor([[0.0, 0.0, tz]]), focal, H, W


def _orientation():
    # on a 16 x 8 image (2:1, y spans [-2, 2]): face 0 at +X +Y, face 1 at -X -Y
    inp = _flat([[0.3, 0.4, 0], [0.9, 0.4, 0], [0.6, 1.6, 0], [-0.9, -1.6, 0], [-0.3, -1.6, 0], [-0.6, -0.4, 0]], H=16, W=8)

    def check(p2f, zbuf, bary):
        rows, cols = torch.nonzero(p2f[0] == 0, as_tuple=True)
        assert rows.numel() > 0 and int(cols.max()) < 4 and int(rows.max()) < 8          # +X -> left columns, +Y -> top rows
        rows, cols = torch.nonzero(p2f[0] == 1, as_tuple=True)
        assert rows.numel() > 0 and int(cols.min()) >= 4 and int(rows.min()) >= 8
    return inp, check


def _edges_and_vertices():
    # 8 x 8: pixel centres at NDC +-0.125, +-0.375, ...; the triangle's vertices sit on pixel centres and its three edges pass
    # through pixel centres, where one barycentric is exactly 0: only the centre (0.125, 0.125) is strictly inside.
    inp = _flat([[-0.125, -0.125, 0], [0.625, -0.125, 0], [-0.125, 0.625, 0]])

    def check(p2f, zbuf, bary):
        want = torch.full((1, 8, 8), -1, dtype=torch.int64)
        want[0, 3, 3] = 0                         # x = 0.125 -> column W-1-4, y = 0.125 -> row H-1-4
        assert torch.equal(p2f, want)
        assert float(zbuf[0, 3, 3]) == 1.0 and bool((bary[0, 3, 3] > 0).all())
    return inp, check


def _nearer_wins():
    # face 0 at depth 3, face 1 (same footprint in NDC) at depth 2: face 1 is in front
    t = [[-0.9, -0.9], [0.9, -0.9], [0.0, 0.9]]
    v = [[x * 3, y * 3, 2.0] for x, y in t] + [[x * 2, y * 2, 1.0] for x, y in t]
    inp = _flat(v)

    def check(p2f, zbuf, bary):
        cov = p2f[0] >= 0
        assert int(cov.sum()) > 10 and bool((p2f[0][cov] == 1).all())
        assert torch.allclose(zbuf[0][cov], torch.full_like(zbuf[0][cov], 2.0))
    return inp, check


def _equal_depth_lower_index():
    # three identical faces: equal pz at every covered pixel, the lowest index wins
    t = [[-0.9, -0.9, 0], [0.9, -0.8, 0], [0.1, 0.9, 0]]
    inp = _flat(t + t + t)

    def check(p2f, zbuf, bary):
        cov = p2f[0] >= 0
        assert int(cov.sum()) > 10 and bool((p2f[0][cov] == 0).all())
    return inp, check


def _skipped():
    # face 0: all depths negative (zmax < 0); face 1: zero area (collinear); face 2: |area| <= 1e-8; face 3: a sliver with one
    # vertex behind the camera -- where its barycentrics are all positive, pz < 0 -- so every pixel stays background
    v = [[-0.5, -0.5, -3.0], [0.5, -0.5, -3.0], [0.0, 0.5, -3.0],
         [-0.5, -0.5, 0.0], [0.0, 0.0, 0.0], [0.5, 0.5, 0.0],
         [0.0, 0.0, 0.0], [1e-5, 0.0, 0.0], [0.0, 1e-5, 0.0],
         [-1.6, -1.6, 1.0], [1.6, 1.6, 1.0], [-0.05, 0.05, -1.5]]
    inp = _flat(v, H=16, W=16)

    def check(p2f, zbuf, bary):
        assert bool((p2f == -1).all()) and bool((zbuf == -1).all()) and bool((bary == -1).all())
    return inp, check


HAND_CASES = {"orientation": _orientation, "edges_and_vertices": _edges_and_vertices, "nearer_wins": _nearer_wins,
              "equal_depth_lower_index": _equal_depth_lower_index, "skipped": _skipped}


@pytest.mark.parametrize("name", sorted(HAND_CASES))
def test_oracle_hand_built_cases(name):
    (verts, faces, R, T, focal, H, W), check = HAND_CASES[name]()
    check(*rp.rasterize(verts, faces, R, T, focal, H, W))


def test_pz_below_zero_is_what_removes_pixels_in_the_skipped_case():
    """Face 3 of the `skipped` case: pixels that pass the inside test but have pz < 0 exist, and none of them is covered."""
    (verts, faces, R, T, focal, H, W), _ = _skipped()
    xn, yn, zn = rp.project(verts, R, T, focal)
    tri = [a[0, faces[3, k]] for k in range(3) for a in (xn, yn, zn)]
    yi, xi = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    px, py = rp.pix_to_ndc(W - 1 - xi, W, H, verts), rp.pix_to_ndc(H - 1 - yi, H, W, verts)
    cov, w0, w1, w2, pz = rp.pixel_test(px, py, *(t.expand_as(px) for t in tri))
    behind = (w0 > 0) & (w1 > 0) & (w2 > 0) & (pz < 0)
    assert int(behind.sum()) > 0 and not bool((cov & behind).any())
    p2f, _, _ = rp.rasterize(verts, faces, R, T, focal, H, W)
    assert not bool((p2f[0] >= 0)[behind].any())


def test_depth_key_orders_like_depth_and_ties_go_to_the_lower_face():
    """The z-buffer key (bits(pz) << 32) | face: -0.0 is canonicalised to +0.0, so pz = -0.0 and +0.0 tie and the lower face
    wins.  (A covered pixel cannot have pz = -0.0 through the projection -- that needs all depths -0.0, i.e. infinite NDC
    coordinates -- so the tie is checked on the key itself.)"""
    pz = torch.tensor([-0.0, 0.0, 0.0, -0.0, 1e-30, 0.5, 0.5, 2.0])
    face = torch.tensor([1, 2, 3, 0, 0, 7, 6, 0])
    key = rp.depth_key(pz, face)
    assert int(key.argmin()) == 3
    assert bool((key[:4].sort().values == rp.depth_key(torch.zeros(4), torch.tensor([0, 1, 2, 3]))).all())
    assert torch.equal(key[4:].argsort(), torch.tensor([0, 2, 1, 3]))


def test_fp64_evaluation_agrees_on_the_hand_built_cases():
    for name, make in HAND_CASES.items():
        (verts, faces, R, T, focal, H, W), check = make()
        check(*rp.rasterize(verts, faces, R, T, focal, H, W, dtype=torch.float64))


def test_package_refuses_without_a_device(monkeypatch):
    raster = importlib.import_module("3dhumangan_b200.raster")
    (verts, faces, R, T, focal, H, W), _ = _orientation()
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    with pytest.raises(RuntimeError):
        raster.rasterize(verts, faces, R, T, focal, H, W)
    with pytest.raises(RuntimeError):
        raster.rasterize_labels(verts, faces, torch.zeros(faces.shape[0], dtype=torch.long), verts[0], R, T, focal, H, W)
    pre = raster.SHHQPreprocessor(gen_height=16, gen_width=8)
    data = {"scales": torch.ones(1), "vertices": verts}
    with pytest.raises(RuntimeError):
        pre(data, rotate=True, h_stddev=0.4, v_stddev=0.1, h_mean=0, v_mean=0)


def test_preprocessor_surface_matches_the_reference():
    """Constructor, buffers (names, shapes, dtypes: the state_dict round-trips with the oracle's, which mirrors
    preprocessor.py:16-34) and the refusal of coordinate_mode='fix_camera'."""
    raster = importlib.import_module("3dhumangan_b200.raster")
    pre = raster.SHHQPreprocessor(gen_height=512, gen_width=256, coordinate_mode="fix_body", h_stddev=0.4)
    ref = rp.SHHQPreprocessor(gen_height=512, gen_width=256)
    sd, rsd = pre.state_dict(), ref.state_dict()
    assert list(sd) == list(rsd) == ["vertex_approximation", "smpl_faces", "smpl_faces_to_labels"]
    for k in sd:
        assert sd[k].shape == rsd[k].shape and sd[k].dtype == rsd[k].dtype
    syn = importlib.import_module("3dhumangan_b200.synthetic")
    mesh = syn.make_body_mesh(0)
    ref.init_smpl(mesh["faces"], mesh["faces_to_labels"])
    pre.load_state_dict(ref.state_dict(), strict=True)
    assert torch.equal(pre.smpl_faces, mesh["faces"]) and torch.equal(pre.smpl_faces_to_labels, mesh["faces_to_labels"])
    with pytest.raises(RuntimeError):
        pre.init_smpl(mesh["faces"] + 6890, mesh["faces_to_labels"])
    with pytest.raises(RuntimeError):
        raster.SHHQPreprocessor(gen_height=512, gen_width=256, coordinate_mode="fix_camera")


def test_body_mesh_has_smpl_counts_and_is_closed():
    syn = importlib.import_module("3dhumangan_b200.synthetic")
    mesh = syn.make_body_mesh(0)
    f = mesh["faces"]
    assert mesh["vertices"].shape == (6890, 3) and f.shape == (13776, 3) and f.dtype == torch.int64
    assert int(f.min()) == 0 and int(f.max()) == 6889
    edges = set(map(tuple, torch.cat([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]]).tolist()))
    assert len(edges) == 3 * 13776 and all((b, a) in edges for a, b in edges)       # closed, consistently oriented
    assert set(mesh["faces_to_labels"].tolist()) == set(range(24))
    assert torch.equal(syn.make_body_mesh(0)["vertices"], mesh["vertices"])
    s = mesh["smpl"]
    assert s["shapedirs"].shape == (6890, 3, 10) and s["posedirs"].shape == (207, 6890 * 3) and s["J_regressor"].shape == (24, 6890)
    assert torch.allclose(s["lbs_weights"].sum(1), torch.ones(6890)) and torch.allclose(s["J_regressor"].sum(1), torch.ones(24))
