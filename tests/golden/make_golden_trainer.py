"""Fixtures for tests/test_cpu_trainer_pin.py: what the UNMODIFIED reference's trainer-side code computes on the recipes below.

  * `PhaseTrainer.init_optimizer` (phase_trainer.py:57-76): the five Adam groups of the generator and the discriminator's group,
    parameters recorded by their names in this package's modules (same names by the state_dict contract);
  * `ExponentialMovingAverage` (lib/components/ema.py:29-48) over 12 seeded parameter moves of the tiny generator: num_updates
    after every update, and per shadow tensor a fixed seeded sample of its elements plus its float64 sum and sum of squares
    (the whole shadow set is 20 MB);
  * `PhaseTrainer._calculate_r1_regularization` (phase_trainer.py:259-294) on a small differentiable stand-in discriminator;
  * `PhaseTrainer._train_discriminator` / `_train_generator` (phase_trainer.py:344-560) on stand-in networks;
  * `extract_metadata` / `get_config` (configs/__init__.py) on every shipped curriculum of configs/map3d.py;
  * bias_act's `activation_funcs` table (lib/components/ops/bias_act.py:22-32).

    HG_REFERENCE=<reference checkout> python tests/golden/make_golden_trainer.py   # writes tests/golden/trainer_pins.{json,npz}
"""
import copy
import importlib
import json
import os
import sys
import tempfile
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))

# ---------------------------------------------------------------------------------------------------------------------------
# recipes (shared with the test)
# ---------------------------------------------------------------------------------------------------------------------------
OPT_META = dict(gen_lr=2e-5, disc_lr=2e-4, betas=(0.0, 0.9),      # (0, 0.9) in configs/map3d.py; this torch wants two floats
                weight_decay=0, appearance_codes_lr_mul=3.0, mapping_net_lr_mul=0.5, neural_field_lr_mul=0.25)
EMA_DECAY, EMA_STEPS, EMA_SAMPLE = 0.999, 12, 16
R1_LAMBDAS = [1.0, 0.0]
COMPOSITION = [(0.0, False), (0.0, True), (1.0, True)]
CURRICULA = ["MAP3DBN", "MAP3DBN512", "MAP3DBN512L"]
GET_CONFIG = [("", 0), ("lr", 0), ("lr", 3), ("map3d_mode", 0), ("map3d_mode", 2)]
GET_CONFIG_NAME = "MAP3DBN512"


def modules(pkg):
    """The tiny generator / discriminator of this package (torch.manual_seed(0)) and their config."""
    gen = importlib.import_module("3dhumangan_b200.modules.generator")
    disc = importlib.import_module("3dhumangan_b200.modules.discriminator")
    cfg = pkg.configs.baseline_config("tiny")
    torch.manual_seed(0)
    return gen.Map3DGenerator(**cfg), disc.UNetDiscriminator(**cfg), cfg


def ema_run(params, make_ema):
    """Seeded starting values for `params`, an EMA built on them, then EMA_STEPS seeded moves each followed by `update`
    (the num_updates ramp (1+n)/(10+n) and the plateau).  -> the EMA and num_updates after every update."""
    gen = torch.Generator().manual_seed(3)
    with torch.no_grad():
        for p in params:
            p.copy_(torch.randn(p.shape, generator=gen) * 0.1)
    ema = make_ema(params)
    counts = []
    for _ in range(EMA_STEPS):
        with torch.no_grad():
            for p in params:
                p.add_(torch.randn(p.shape, generator=gen) * 0.01)
        ema.update(params)
        counts.append(ema.num_updates)
    return ema, counts


def ema_summary(tensors):
    """-> (fixed seeded sample of up to EMA_SAMPLE elements of every tensor, concatenated; [sum, sum of squares] per tensor)."""
    sample, moments = [], []
    for i, t in enumerate(tensors):
        flat = t.detach().reshape(-1)
        idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(i))[:EMA_SAMPLE]
        sample.append(flat[idx])
        moments.append([float(flat.double().sum()), float(flat.double().square().sum())])
    return torch.cat(sample), torch.tensor(moments, dtype=torch.float64)


class R1Scaler:
    """GradScaler's two calls used by the R1 penalty, with a non-trivial scale."""

    def scale(self, t):
        return t * 1024.0

    def get_scale(self):
        return 1024.0


def r1_run(penalty, gan_lambda):
    """`penalty(x, out, scaler, meta)` on a small differentiable stand-in for the discriminator, then backward (the double
    backward).  -> (value, gradient of the first conv weight, gradient of the segmentation conv weight)."""
    g = torch.Generator().manual_seed(9)
    w1 = torch.randn(6, 3, 3, 3, generator=g, dtype=torch.float64) * 0.3
    w2 = torch.randn(5, 6, 1, 1, generator=g, dtype=torch.float64) * 0.3
    x0 = torch.randn(3, 3, 8, 8, generator=g, dtype=torch.float64)
    meta = dict(gan_lambda=gan_lambda, segmentation_lambda=1.0, r1_lambda=0.25)
    a, b = w1.clone().requires_grad_(True), w2.clone().requires_grad_(True)
    x = x0.clone().requires_grad_(True)
    h = torch.nn.functional.leaky_relu(torch.nn.functional.conv2d(x, a, padding=1), 0.2)
    seg = torch.nn.functional.conv2d(torch.tanh(h), b)
    out = {"prediction": (h * h).mean(dim=(1, 2, 3)), "segments": seg}
    pen = penalty(x, out, R1Scaler(), meta)
    pen.backward()
    return float(pen), a.grad.clone(), b.grad.clone() if b.grad is not None else torch.zeros_like(b)


class StandInG(torch.nn.Module):
    """A generator with the call signature the trainer uses (z, conditions, latent_indices=..., **meta) -> {'rgbs', 'rgbs_render'}."""

    def __init__(self, L):
        super().__init__()
        g = torch.Generator().manual_seed(21)
        self.neural_field_mapping_network = torch.nn.Linear(L, 6)
        self.synthesis_network = torch.nn.Conv2d(6, 3, 3, padding=1)
        with torch.no_grad():
            for p in self.parameters():
                p.copy_(torch.randn(p.shape, generator=g) * 0.3)

    def forward(self, z, conditions, latent_indices=None, disable_synthesis=False, **kwargs):
        h = torch.tanh(self.neural_field_mapping_network(z))[:, :, None, None] + conditions["x"]
        rgb = torch.tanh(self.synthesis_network(h))
        return {"rgbs": rgb, "rgbs_render": torch.nn.functional.avg_pool2d(rgb, 2)}


class StandInD(torch.nn.Module):
    def __init__(self, label_dim):
        super().__init__()
        g = torch.Generator().manual_seed(22)
        self.c1 = torch.nn.Conv2d(3, 8, 3, padding=1)
        self.seg = torch.nn.Conv2d(8, label_dim, 1)
        self.pred = torch.nn.Linear(8, 1)
        self.step = 0
        with torch.no_grad():
            for p in self.parameters():
                p.copy_(torch.randn(p.shape, generator=g) * 0.3)

    def forward(self, x, conditions, alpha=1.0, mode="real", **kwargs):
        h = torch.nn.functional.leaky_relu(self.c1(x), 0.2) + (0.1 if mode == "real" else -0.1) * conditions["x"][:, :1]
        return {"prediction": self.pred(h.mean(dim=(2, 3))), "segments": self.seg(h), "latents": h.mean(dim=(2, 3))}


def composition_case(gan_lambda, do_r1):
    """-> (latent dim, label dim, meta, phase, images, labels, x, z_d, z_g) of one D step + G step on the stand-ins."""
    L, LD, B, H = 5, 7, 4, 8
    phase = {"name": "uncond", "uncond": True, "rotate": True, "gen_modal": "rgbs", "do_r1": do_r1}
    meta = dict(latent_dim=L, label_dim=LD, z_dist="gaussian", gan_lambda=gan_lambda, segmentation_lambda=1.0, latent_lambda=0,
                perceptual_lambda=[0, 0, 0, 0], photometric_lambda=0, r1_lambda=0.25, grad_clip=1e9, gen_lr=0.0, disc_lr=0.0,
                betas=(0.0, 0.9), weight_decay=0, appearance_codes_lr_mul=1.0, mapping_net_lr_mul=1.0, neural_field_lr_mul=1.0,
                batch_split=2, phases=[phase], render_height=4, render_width=4, gen_height=H, gen_width=H)
    g = torch.Generator().manual_seed(23)
    images = torch.randn(B, 3, H, H, generator=g).clamp_(-1, 1)
    labels = torch.randint(0, LD, (B, H, H), generator=g)
    x = torch.randn(B, 6, H, H, generator=g) * 0.2
    z_d, z_g = torch.randn(B, L, generator=g), torch.randn(B, L, generator=g)
    return L, LD, meta, phase, images, labels, x, z_d, z_g


def composition_key(gan_lambda, do_r1):
    return f"composition_{gan_lambda}_{int(do_r1)}"


def curriculum_steps(cur):
    """Steps on both sides of every schedule boundary of a curriculum."""
    return sorted({0, 1, 999, 1000, 200000, 200001, 300000, 300001, 300002, 10 ** 6} | {int(k) for k in cur if isinstance(k, int)} |
                  {int(k) + 1 for k in cur if isinstance(k, int)})


# JSON cannot tell a tuple from a list, nor hold a class: both are tagged so that the test compares with `==` as before
def encode(v):
    if isinstance(v, tuple):
        return {"__tuple__": [encode(x) for x in v]}
    if isinstance(v, list):
        return [encode(x) for x in v]
    if isinstance(v, dict):
        return {k: encode(x) for k, x in v.items()}
    if isinstance(v, type):
        return {"__class__": v.__name__}
    if isinstance(v, np.generic):
        return v.item()
    return v


def decode_hook(d):
    """json.load object_hook: tuples back to tuples, classes to their names."""
    if set(d) == {"__tuple__"}:
        return tuple(d["__tuple__"])
    if set(d) == {"__class__"}:
        return d["__class__"]
    return d


# ---------------------------------------------------------------------------------------------------------------------------
# recording
# ---------------------------------------------------------------------------------------------------------------------------
def main():
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "oracle", "shims"))
    sys.path.insert(0, os.environ["HG_REFERENCE"])
    pkg = importlib.import_module("3dhumangan_b200")
    pt = importlib.import_module("lib.trainers.phase_trainer")
    ema_ref = importlib.import_module("lib.components.ema")
    ref_cfg = importlib.import_module("configs")
    ba = importlib.import_module("lib.components.ops.bias_act")
    js, arrays = {}, {}

    G, D, cfg = modules(pkg)
    with tempfile.TemporaryDirectory() as ckpt:            # no checkpoint to resume from
        me = types.SimpleNamespace(generator_ddp=G, discriminator_ddp=D, output_dir=ckpt, device="cpu")
        pt.PhaseTrainer.init_optimizer(me, dict(cfg, **OPT_META))
    gname = {id(p): n for n, p in G.named_parameters()}
    dname = {id(p): n for n, p in D.named_parameters()}
    js["optimizer_G"] = [{"name": g["name"], "lr": g["lr"], "betas": list(g["betas"]), "weight_decay": g["weight_decay"], "eps": g["eps"],
                          "params": [gname[id(p)] for p in g["params"]]} for g in me.optimizer_G.param_groups]
    js["optimizer_D"] = [{"lr": g["lr"], "betas": list(g["betas"]), "params": [dname[id(p)] for p in g["params"]]}
                         for g in me.optimizer_D.param_groups]

    G, _, _ = modules(pkg)
    ema, counts = ema_run(list(G.parameters()), lambda ps: ema_ref.ExponentialMovingAverage(ps, decay=EMA_DECAY))
    js["ema_num_updates"] = counts
    js["ema_shadow_count"] = len(ema.shadow_params)
    arrays["ema_sample"], arrays["ema_moments"] = ema_summary(ema.shadow_params)

    for gl in R1_LAMBDAS:
        pen, ga, gb = r1_run(lambda x, out, scaler, meta: pt.PhaseTrainer._calculate_r1_regularization(
            types.SimpleNamespace(scaler=scaler, amp=False), x, out, {"do_r1": True}, meta), gl)
        arrays[f"r1_{gl}_value"], arrays[f"r1_{gl}_grad_a"], arrays[f"r1_{gl}_grad_b"] = torch.tensor(pen, dtype=torch.float64), ga, gb

    for gl, do_r1 in COMPOSITION:
        L, LD, meta, phase, images, labels, x, z_d, z_g = composition_case(gl, do_r1)
        Gr, Dr = StandInG(L), StandInD(LD)
        me = types.SimpleNamespace(amp=False, device="cpu", batch_split=2, rank=0, generator_ddp=Gr, discriminator_ddp=Dr, discriminator=Dr,
                                   scaler=torch.amp.GradScaler("cuda", enabled=False))
        for name in ("_train_discriminator", "_train_generator", "_get_disc_input_real", "_get_disc_input_gen",
                     "_calculate_r1_regularization", "_calculate_segmentation_loss"):
            setattr(me, name, types.MethodType(getattr(pt.PhaseTrainer, name), me))
        zs = [z_d, z_g]
        saved = pt.z_sampler, pt.training_stats.report
        pt.z_sampler = lambda *a, **k: zs.pop(0)
        pt.training_stats.report = lambda *a, **k: None
        try:
            data = {"images": images, "body_segments": labels, "rasterized_segments": labels, "latents": torch.zeros(images.shape[0], L), "x": x}
            d_ref = me._train_discriminator(data, 1.0, meta, phase)
            d_ref.backward()
            dgrads = [p.grad.clone() for p in Dr.parameters()]
            Gr.zero_grad()
            Dr.zero_grad()
            g_ref, _ = me._train_generator(data, 1.0, meta, phase)
            ggrads = [p.grad.clone() for p in Gr.parameters()]
        finally:
            pt.z_sampler, pt.training_stats.report = saved
        key = composition_key(gl, do_r1)
        arrays[key + "_d_loss"] = torch.tensor(float(d_ref), dtype=torch.float64)
        arrays[key + "_g_loss"] = torch.tensor(float(g_ref), dtype=torch.float64)
        for i, t in enumerate(dgrads):
            arrays[f"{key}_d_grad_{i}"] = t
        for i, t in enumerate(ggrads):
            arrays[f"{key}_g_grad_{i}"] = t
        for i, p in enumerate(list(Gr.parameters()) + list(Dr.parameters())):
            arrays[f"{key}_param_{i}"] = p.detach()

    js["curricula"] = {}            # per curriculum: the distinct metadata dicts, and for every step the index of its dict
    for name in CURRICULA:
        cur = getattr(ref_cfg, name)
        metas, steps = [], []
        for step in curriculum_steps(cur):
            m = encode(ref_cfg.extract_metadata(cur, step))
            if m not in metas:
                metas.append(m)
            steps.append([step, metas.index(m)])
        js["curricula"][name] = {"metadata": metas, "steps": steps}

    js["get_config"] = []
    for tune, variant in GET_CONFIG:
        saved = copy.deepcopy(getattr(ref_cfg, GET_CONFIG_NAME))
        try:
            a = ref_cfg.get_config(types.SimpleNamespace(config=GET_CONFIG_NAME, tune=tune, variant=variant))
            js["get_config"].append({"tune": tune, "variant": variant, "name": a["name"], "map3d_mode": a["map3d_mode"],
                                     "neural_field_cls": a["neural_field_cls"].__name__,
                                     "stages": [[k, encode(a[k])] for k in a if isinstance(k, int)]})
        finally:
            setattr(ref_cfg, GET_CONFIG_NAME, saved)

    js["activations"] = {k: [v.cuda_idx, float(v.def_alpha), float(v.def_gain), v.ref, v.has_2nd_grad]
                         for k, v in ba.activation_funcs.items() if v.cuda_idx is not None}

    with open(os.path.join(HERE, "trainer_pins.json"), "w") as f:
        json.dump(js, f, indent=1)
    np.savez_compressed(os.path.join(HERE, "trainer_pins.npz"), **{k: v.numpy() for k, v in arrays.items()})
    print("written", len(js), "json entries,", len(arrays), "arrays")


if __name__ == "__main__":
    main()
