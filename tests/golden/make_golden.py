"""Generate golden fixtures by running the UNMODIFIED reference (build container only).

    python tests/golden/make_golden.py            # writes tests/golden/*.npz

Needs /root/reference plus the test-only shims in oracle/shims (pytorch3d / smplx are not in this
image).  Parameters come from `oracle.port.init_*_params(seed)` and are loaded into the
reference modules with a strict `load_state_dict`, inputs from `synthetic.make_conditions`,
random draws from a seeded global torch RNG (the reference draws them itself; the fixture stores
the seed, and `rng.draw_render_noise` replays the identical sequence for the oracle / kernels).
Fixtures hold only small OUTPUT tensors + the recipe (seeds, config overrides).
"""
import copy
import importlib
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("HG_REFERENCE", "/root/reference")

CASES = {
    # name: (base BASELINE config, overrides, param seed, sigma_gain, sigma_bias, batch, noise_std)
    "g_tiny_mixed": ("C2", dict(gen_height=32, gen_width=32, render_height=8, render_width=8), 0, 1.0, 0.0, 2, 0.0),
    "g_tiny_dense": ("C2", dict(gen_height=32, gen_width=32, render_height=8, render_width=8), 3, 200.0, 1.0, 2, 0.5),
    "g_tiny_portrait": ("C2", dict(gen_height=64, gen_width=32, render_height=12, render_width=6, num_steps=16), 4, 200.0, 1.0, 1, 0.0),
    "g_small_isolated_legacy": ("C2", dict(gen_height=32, gen_width=32, render_height=8, render_width=8, hidden_dim=64,
                                            latent_dim=64, feature_dim=64, map3d_mode="isolated", legacy_mode=True,
                                            last_back=True), 5, 200.0, 1.0, 2, 0.0),
    # the widths of the other two shipped curricula: MAP3DBN512L (420, isolated + legacy, the released checkpoint, with the
    # sample app's last_back) and MAP3DBN (384, mixed) -- configs/map3d.py:194-290, :3-95
    "g_h420_isolated_legacy": ("C2", dict(gen_height=32, gen_width=32, render_height=8, render_width=8, hidden_dim=420,
                                           latent_dim=420, feature_dim=420, map3d_mode="isolated", legacy_mode=True,
                                           last_back=True), 6, 200.0, 1.0, 2, 0.0),
    "g_h384_mixed": ("C2", dict(gen_height=32, gen_width=16, render_height=8, render_width=4, hidden_dim=384, latent_dim=384,
                                 feature_dim=384), 7, 200.0, 1.0, 2, 0.5),
}
D_CASES = {"d_tiny": (dict(gen_height=64, gen_width=64), 7, 2)}
# the g_tiny_dense recipe drawn at a second seed: the reference's own draws, which tests/test_oracle_pin.py replays through
# `rng.draw_render_noise` (stored as <case>_seed<seed>.npz: rgbs, and of the feature maps every 17th element + the L2 norm)
REPLAY = ("g_tiny_dense", 77)


def reference_modules():
    sys.path.insert(0, os.path.join(ROOT, "oracle", "shims"))
    sys.path.insert(0, REF)
    import lib.generators, lib.discriminators, lib.implicit_funcitions  # noqa
    return sys.modules["lib.generators"], sys.modules["lib.discriminators"], sys.modules["lib.implicit_funcitions"]


def build_case(pkg, port, name):
    base, over, pseed, sg, sb, B, noise_std = CASES[name]
    cfg = pkg.configs.baseline_config(base)
    cfg.update(over)
    cfg["nerf_noise"] = noise_std
    params = port.init_generator_params(cfg, seed=pseed, sigma_gain=sg, sigma_bias=sb)
    cond = pkg.synthetic.make_conditions(B, seed=11 + pseed)
    z = torch.randn(B, cfg["latent_dim"], generator=torch.Generator().manual_seed(100 + pseed))
    return cfg, params, cond, z, B


def run_reference_generator(gens, impl, cfg, params, cond, z, seed):
    meta = dict(cfg)
    meta["neural_field_cls"] = getattr(impl, meta["neural_field_cls"])
    G = gens.Map3DGenerator(**meta)
    G.load_state_dict(params, strict=True)
    G.set_device("cpu")
    G.train()
    torch.manual_seed(seed)
    with torch.no_grad():
        rr, fmap, depth, w, _ = G.render(*G.neural_field_mapping_network(torch.zeros_like(z) if not meta.get("neural_field_latent_input", True) else z),
                                         cond, coarse_steps=meta["num_steps"], fine_steps=meta["num_steps"], **meta)
    torch.manual_seed(seed)
    with torch.no_grad():
        out = G(z, cond, **meta)
    sd = G.state_dict()
    return out, fmap, depth, sd


def main():
    sys.path.insert(0, ROOT)
    pkg = importlib.import_module("3dhumangan_b200")
    from oracle import port
    gens, discs, impl = reference_modules()
    only = [a for a in sys.argv[1:] if not a.startswith("-")]          # optional: regenerate just these cases
    manifest = {}
    if only:
        with open(os.path.join(HERE, "manifest.json")) as f:
            manifest = json.load(f)
    for name in CASES:
        if only and name not in only:
            continue
        cfg, params, cond, z, B = build_case(pkg, port, name)
        seed = 1234
        out, fmap, depth, sd = run_reference_generator(gens, impl, cfg, copy.deepcopy(params), cond, z, seed)
        blk = "synthesis_network.network.m3d_0."
        np.savez_compressed(os.path.join(HERE, name + ".npz"),
                            rgbs=out["rgbs"].numpy(), rgbs_render=out["rgbs_render"].numpy(),
                            feature_maps=fmap.numpy(), depths=depth.numpy(),
                            running_mean0=sd[blk + "spade_0.first_norm.running_mean"].numpy(),
                            running_var0=sd[blk + "spade_0.first_norm.running_var"].numpy(),
                            weight_u0=sd[blk + "conv_0.weight_u"].numpy())
        manifest[name] = {"rng_seed": seed, "recipe": [CASES[name][0], CASES[name][1], *CASES[name][2:]]}
        print(name, "rgbs", tuple(out["rgbs"].shape), float(out["rgbs"].abs().mean()))
    name, seed = REPLAY
    if not only or f"{name}_seed{seed}" in only:
        cfg, params, cond, z, B = build_case(pkg, port, name)
        out, fmap, _, _ = run_reference_generator(gens, impl, cfg, copy.deepcopy(params), cond, z, seed)
        np.savez_compressed(os.path.join(HERE, f"{name}_seed{seed}.npz"), rgbs=out["rgbs"].numpy(),
                            feature_maps_every17=fmap.reshape(-1)[::17].numpy(), feature_maps_norm=np.array(float(fmap.double().norm())))
        print(f"{name}_seed{seed}", "rgbs", tuple(out["rgbs"].shape))
    for name, (over, pseed, B) in D_CASES.items():
        if only and name not in only:
            continue
        cfg = pkg.configs.baseline_config("C2")
        cfg.update(over)
        params = port.init_discriminator_params(cfg, seed=pseed)
        D = discs.UNetDiscriminator(**cfg)
        D.load_state_dict(params, strict=True)
        D.train()
        img = torch.randn(B, 3, cfg["gen_height"], cfg["gen_width"], generator=torch.Generator().manual_seed(pseed)).clamp(-1, 1)
        with torch.no_grad():
            o = D(img, None, alpha=1.0)
        np.savez_compressed(os.path.join(HERE, name + ".npz"), prediction=o["prediction"].numpy(),
                            latents=o["latents"].numpy(), segments=o["segments"].numpy())
        manifest[name] = {"recipe": [over, pseed, B]}
        print(name, "pred", tuple(o["prediction"].shape))
    with open(os.path.join(HERE, "manifest.json"), "w") as f:
        json.dump(manifest, f, indent=1)


if __name__ == "__main__":
    main()
