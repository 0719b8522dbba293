"""The preprocessor's rasteriser on the device (3dhumangan_b200/raster.py, csrc/raster.cu) against the oracle evaluated on the
device (oracle/raster_port.py, pinned to the reference's own preprocessor code by tests/test_cpu_raster_pin.py)."""
import importlib
import importlib.util
import math
import os

import pytest
import torch

from oracle import raster_port as rp

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROT = dict(h_stddev=0.4, v_stddev=0.1, h_mean=0, v_mean=0)            # the three curricula's view distribution


def _mod(name):
    return importlib.import_module("3dhumangan_b200." + name)


def _cpu_cases():
    spec = importlib.util.spec_from_file_location("test_cpu_raster_pin", os.path.join(HERE, "test_cpu_raster_pin.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.HAND_CASES


def _posed_body(B, seed):
    """-> (mesh, data dict on the device from smpl.lbs + conditions_fix_body on the synthetic body)."""
    smpl, syn = _mod("smpl"), _mod("synthetic")
    mesh = syn.make_body_mesh(0)
    model = smpl.SMPLModel.from_arrays(**mesh["smpl"], device="cuda")
    g = torch.Generator().manual_seed(seed)
    out = smpl.lbs(torch.randn(B, 10, generator=g) * 0.5, torch.randn(B, 24, 3, generator=g) * 0.3, model)
    orig_cam = torch.stack([1.2 + 0.2 * torch.rand(B, generator=g), torch.ones(B), 0.1 * torch.randn(B, generator=g),
                            0.1 * torch.randn(B, generator=g)], 1)
    return mesh, smpl.conditions_fix_body(orig_cam, out, model)


def _views(data, seed):
    """Seeded rotate=True views -> (R_raster, T_raster) as the preprocessor builds them."""
    smpl, raster = _mod("smpl"), _mod("raster")
    B = data["scales"].shape[0]
    g = torch.Generator().manual_seed(seed)
    h, v = torch.randn(B, generator=g) * ROT["h_stddev"], torch.randn(B, generator=g) * ROT["v_stddev"]
    R = torch.inverse(smpl.body_rotation(data, h, v, torch.zeros(B)))
    T = data["T"][:, :3, -1].clone()
    T[:, -1] = raster.FOCAL_RASTER / data["scales"] * 0.5
    return R, T


def _oracle_labels(p2f, faces, labels, sem_verts, bary):
    """preprocessor.py:156-174 on per-mesh face indices."""
    bg = p2f < 0
    f = p2f.clamp_min(0)
    seg = torch.where(bg, 1, labels[f] + 2)
    vert = torch.gather(faces[f], -1, torch.argmax(bary, -1, keepdim=True))[..., 0]
    sem = torch.where(bg[..., None], 0.0, sem_verts[vert]).permute(0, 3, 1, 2)
    return seg, sem


@pytest.mark.parametrize("H,W", [(256, 128), (512, 256), (512, 512)])
def test_kernel_matches_oracle_bitwise_on_the_posed_body(H, W):
    raster = _mod("raster")
    mesh, data = _posed_body(4, seed=30 + H + W)
    R, T = _views(data, seed=H + W)
    faces, labels = mesh["faces"].cuda(), mesh["faces_to_labels"].cuda()
    sem_verts = data["tpose_vertices"][0]
    F = faces.shape[0]
    p2f, zbuf, bary = raster.rasterize(data["vertices"], faces, R, T, -raster.FOCAL_RASTER, H, W)
    seg, sem = raster.rasterize_labels(data["vertices"], faces, labels, sem_verts, R, T, -raster.FOCAL_RASTER, H, W)
    rf, rz, rb = rp.rasterize(data["vertices"], faces, R, T, -raster.FOCAL_RASTER, H, W)
    torch.cuda.synchronize()
    off = torch.arange(4, device="cuda")[:, None, None] * F
    assert torch.equal(p2f, torch.where(rf >= 0, rf + off, rf))
    assert torch.equal(zbuf, rz) and torch.equal(bary, rb)
    rseg, rsem = _oracle_labels(rf, faces, labels, sem_verts, rb)
    assert torch.equal(seg, rseg) and torch.equal(sem, rsem)
    cov = rf >= 0
    assert int(cov.sum()) > 0.05 * cov.numel() and len(set(seg.unique().tolist())) > 12
    f64, _, _ = rp.rasterize(data["vertices"], faces, R, T, -raster.FOCAL_RASTER, H, W, dtype=torch.float64)
    changed = int(((f64 != rf) & (cov | (f64 >= 0))).sum())
    print(f"\n{H}x{W} B=4: {int(cov.sum())} covered pixels, {changed} change face when the oracle is evaluated in fp64")


@pytest.mark.parametrize("name", ["orientation", "edges_and_vertices", "nearer_wins", "equal_depth_lower_index", "skipped"])
def test_kernel_hand_built_cases(name):
    raster = _mod("raster")
    (verts, faces, R, T, focal, H, W), check = _cpu_cases()[name]()
    out = raster.rasterize(verts.cuda(), faces.cuda(), R.cuda(), T.cuda(), focal, H, W)
    ref = rp.rasterize(verts, faces, R, T, focal, H, W)
    out = [t.cpu() for t in out]
    check(*out)
    for a, b in zip(out, ref):
        assert torch.equal(a, b)


def test_deterministic_and_batch_independent():
    raster = _mod("raster")
    mesh, data = _posed_body(16, seed=40)
    R, T = _views(data, seed=41)
    faces = mesh["faces"].cuda()
    F = faces.shape[0]
    a = raster.rasterize(data["vertices"], faces, R, T, -raster.FOCAL_RASTER, 512, 512)
    b = raster.rasterize(data["vertices"], faces, R, T, -raster.FOCAL_RASTER, 512, 512)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    for i in (0, 7, 15):
        one = raster.rasterize(data["vertices"][i:i + 1], faces, R[i:i + 1], T[i:i + 1], -raster.FOCAL_RASTER, 512, 512)
        p = a[0][i]
        assert torch.equal(torch.where(p >= 0, p - i * F, p), one[0][0])
        assert torch.equal(a[1][i], one[1][0]) and torch.equal(a[2][i], one[2][0])


def test_preprocessor_matches_oracle_preprocessor():
    raster, smpl = _mod("raster"), _mod("smpl")
    mesh, data = _posed_body(3, seed=50)
    for H, W in ((256, 128), (512, 256)):
        pre = raster.SHHQPreprocessor(gen_height=H, gen_width=W).cuda()
        pre.init_smpl(mesh["faces"], mesh["faces_to_labels"])
        ref = rp.SHHQPreprocessor(gen_height=H, gen_width=W).cuda()
        ref.load_state_dict(pre.state_dict(), strict=True)
        torch.manual_seed(51)
        out = pre(dict(data), rotate=True, **ROT)
        torch.manual_seed(51)
        want = ref(dict(data), rotate=True, **ROT)
        torch.manual_seed(51)
        h, v = torch.randn(3) * ROT["h_stddev"], torch.randn(3) * ROT["v_stddev"]
        torch.cuda.synchronize()
        assert out["rasterized_segments"].dtype == torch.int64 and out["rasterized_semantics"].dtype == torch.float32
        assert torch.equal(out["rasterized_segments"], want["rasterized_segments"])
        assert torch.equal(out["rasterized_semantics"], want["rasterized_semantics"])
        assert torch.equal(out["cam2world_matrices"], smpl.cam2world_fix_body(data, h, v, torch.zeros(3)))


def test_end_to_end_training_iteration_on_rasterised_labels(pkg):
    raster, smpl = _mod("raster"), _mod("smpl")
    gen, disc, ts = _mod("modules.generator"), _mod("modules.discriminator"), _mod("train_step")
    cfg = pkg.configs.baseline_config("tiny")
    cfg.update(gen_height=64, gen_width=64, render_height=8, render_width=8, num_steps=32, nerf_noise=0.5)
    B = 2
    mesh = _mod("synthetic").make_body_mesh(0)
    model = smpl.SMPLModel.from_arrays(**mesh["smpl"], device="cuda")
    g = torch.Generator().manual_seed(60)
    out = smpl.lbs(torch.randn(B, 10, generator=g) * 0.5, torch.randn(B, 24, 3, generator=g) * 0.3, model)
    cond = smpl.conditions_fix_body(torch.tensor([[1.3, 1.3, 0.0, 0.05]] * B), out, model)
    pre = raster.SHHQPreprocessor(**cfg).cuda()
    pre.init_smpl(mesh["faces"], mesh["faces_to_labels"])
    torch.manual_seed(61)
    data = pre(cond, rotate=True, **cfg)
    labels = data.pop("rasterized_segments")
    data.pop("rasterized_semantics")
    vals = set(labels.unique().tolist())
    assert 1 in vals and vals <= set(range(1, 26)) and len(vals - {1}) > 0
    torch.manual_seed(62)
    G = gen.Map3DGenerator(**cfg).cuda().train()
    G.set_device(torch.device("cuda:0"))
    D = disc.UNetDiscriminator(**cfg).cuda().train()
    t = ts.Trainer(G, D, cfg, amp=False, ddp=False)
    batch = dict(cond=data, images=torch.randn(B, 3, 64, 64, device="cuda").clamp_(-1, 1), labels=labels)
    d, g_ = t.iteration(batch)
    torch.cuda.synchronize()
    assert torch.isfinite(d) and torch.isfinite(g_)


def test_rasterize_captures_into_a_cuda_graph():
    raster = _mod("raster")
    mesh, data = _posed_body(4, seed=70)
    R, T = _views(data, seed=71)
    faces, labels = mesh["faces"].cuda(), mesh["faces_to_labels"].cuda()
    sem_verts = data["tpose_vertices"][0].contiguous()
    args = (data["vertices"], faces, R, T, -raster.FOCAL_RASTER, 512, 256)
    eager = raster.rasterize(*args) + raster.rasterize_labels(data["vertices"], faces, labels, sem_verts, R, T,
                                                              -raster.FOCAL_RASTER, 512, 256)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            cap = raster.rasterize(*args) + raster.rasterize_labels(data["vertices"], faces, labels, sem_verts, R, T,
                                                                    -raster.FOCAL_RASTER, 512, 256)
    torch.cuda.current_stream().wait_stream(s)
    for x in cap:
        x.fill_(7)
    graph.replay()
    torch.cuda.synchronize()
    for a, b in zip(eager, cap):
        assert torch.equal(a, b)


def test_out_of_range_faces_are_refused():
    raster = _mod("raster")
    (verts, faces, R, T, focal, H, W), _ = _cpu_cases()["orientation"]()
    with pytest.raises(RuntimeError):
        raster.rasterize(verts.cuda(), (faces + 100).cuda(), R.cuda(), T.cuda(), focal, H, W)
    with pytest.raises(RuntimeError):
        raster.rasterize(verts.cuda(), faces.cuda(), R.cuda(), T.cuda(), focal, H, W, faces_per_pixel=2)
