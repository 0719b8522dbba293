"""Times the preprocessor's rasteriser on the device and prints one JSON line.

For each image size (B = 16 at 512x512 and 512x256 by default) on the posed synthetic body (`synthetic.make_body_mesh`, SMPL's
6 890 vertices / 13 776 faces, seeded views at the curricula's h_stddev / v_stddev):
  raster_ms       CUDA-event median of `raster.rasterize_labels` (clear + splat + resolve -> segments + semantics)
  preprocess_ms   CUDA-event median of the whole `SHHQPreprocessor.forward(rotate=True)` (view rotation, 3x3 / 4x4 inverses,
                  cam2world, rasteriser)
  bytes           HBM bytes the rasteriser must move: segments (8 B/pixel) + semantics (12 B/pixel) written, the key buffer
                  cleared and read back (16 B/pixel), vertices / faces / labels read once
  raster_gbps     bytes / raster time
The GPU's name and power limit are reported with the numbers.

    python tools/raster_bench.py [--batch 16] [--iters 50] [--sizes 512x512,512x256]"""
import argparse
import importlib
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def median_ms(fn, iters, warmup=5):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(iters):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        e.synchronize()
        times.append(s.elapsed_time(e))
    times.sort()
    return times[len(times) // 2], times[0], times[-1]


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        return out or None
    except (OSError, subprocess.SubprocessError):
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--sizes", default="512x512,512x256")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("raster_bench: no CUDA device")
    raster, smpl, syn = (importlib.import_module("3dhumangan_b200." + m) for m in ("raster", "smpl", "synthetic"))
    B = args.batch
    mesh = syn.make_body_mesh(0)
    model = smpl.SMPLModel.from_arrays(**mesh["smpl"], device="cuda")
    g = torch.Generator().manual_seed(0)
    out = smpl.lbs(torch.randn(B, 10, generator=g) * 0.5, torch.randn(B, 24, 3, generator=g) * 0.3, model)
    orig_cam = torch.stack([1.2 + 0.2 * torch.rand(B, generator=g), torch.ones(B), 0.1 * torch.randn(B, generator=g),
                            0.1 * torch.randn(B, generator=g)], 1)
    cond = smpl.conditions_fix_body(orig_cam, out, model)
    faces, labels = mesh["faces"].cuda(), mesh["faces_to_labels"].cuda()
    V, F = mesh["vertices"].shape[0], faces.shape[0]
    rot = dict(h_stddev=0.4, v_stddev=0.1, h_mean=0, v_mean=0)
    h, v = torch.randn(B, generator=g) * rot["h_stddev"], torch.randn(B, generator=g) * rot["v_stddev"]
    R = torch.inverse(smpl.body_rotation(cond, h, v, torch.zeros(B))).contiguous()
    T = cond["T"][:, :3, -1].clone()
    T[:, -1] = raster.FOCAL_RASTER / cond["scales"] * 0.5
    sem_verts = cond["tpose_vertices"][0].contiguous()
    res = {"metric": "preprocessor_raster", "batch": B, "device": torch.cuda.get_device_name(0), "power_limit": power_limit(),
           "sizes": {}}
    for size in args.sizes.split(","):
        H, W = (int(x) for x in size.split("x"))
        run = lambda: raster.rasterize_labels(cond["vertices"], faces, labels, sem_verts, R, T, -raster.FOCAL_RASTER, H, W)
        seg, _ = run()
        covered = int((seg != 1).sum())
        t_r, t_r_min, t_r_max = median_ms(run, args.iters)
        pre = raster.SHHQPreprocessor(gen_height=H, gen_width=W).cuda()
        pre.init_smpl(mesh["faces"], mesh["faces_to_labels"])
        t_p, t_p_min, t_p_max = median_ms(lambda: pre(dict(cond), rotate=True, **rot), args.iters)
        px = B * H * W
        nbytes = px * (8 + 12) + px * 16 + B * V * 12 + F * 12 + F * 8 + V * 12
        res["sizes"][size] = {"raster_ms": round(t_r, 4), "raster_ms_min": round(t_r_min, 4), "raster_ms_max": round(t_r_max, 4),
                              "preprocess_ms": round(t_p, 4), "preprocess_ms_min": round(t_p_min, 4),
                              "preprocess_ms_max": round(t_p_max, 4), "covered_pixels": covered, "bytes": nbytes,
                              "raster_gbps": round(nbytes / (t_r * 1e-3) / 1e9, 1),
                              "hbm_floor_ms_at_7700_gbps": round(nbytes / 7.7e12 * 1e3, 4)}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
