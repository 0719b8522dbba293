"""Host-side trainer logic pinned against the reference's own code: the five Adam parameter groups of
`PhaseTrainer.init_optimizer` (phase_trainer.py:57-76), the EMA update of `lib/components/ema.py:29-48`, the R1 penalty, the
D-step / G-step composition, the curricula and the bias_act activation table.  The unmodified reference functions were executed
on the recipes of tests/golden/make_golden_trainer.py (on THIS package's modules where parameters matter: same parameter names
by the state_dict contract); tests/golden/trainer_pins.{json,npz} hold what they computed."""
import copy
import importlib.util
import json
import os
import types

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def _load_recipes():
    spec = importlib.util.spec_from_file_location("make_golden_trainer", os.path.join(GOLD, "make_golden_trainer.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


rec = _load_recipes()


@pytest.fixture(scope="module")
def gold():
    with open(os.path.join(GOLD, "trainer_pins.json")) as f:
        js = json.load(f, object_hook=rec.decode_hook)
    arrays = np.load(os.path.join(GOLD, "trainer_pins.npz"))
    js.update({k: torch.from_numpy(arrays[k]) for k in arrays.files})
    return js


def test_optimizer_groups_match_phase_trainer_init_optimizer(pkg, gold):
    ts = importlib.import_module("3dhumangan_b200.train_step")
    G, D, cfg = rec.modules(pkg)
    meta = dict(cfg, **rec.OPT_META)
    og, od = ts.make_optimizers(G, D, meta, fused=False)
    og_f, od_f = ts.make_optimizers(G, D, meta, fused=True)         # the multi-tensor optimiser keeps the same groups
    gname = {id(p): n for n, p in G.named_parameters()}
    dname = {id(p): n for n, p in D.named_parameters()}
    for mine in (og, og_f):
        assert len(mine.param_groups) == len(gold["optimizer_G"]) == 5
        for a, b in zip(mine.param_groups, gold["optimizer_G"]):
            assert a["name"] == b["name"]
            assert a["lr"] == pytest.approx(b["lr"], rel=0, abs=0) and tuple(a["betas"]) == tuple(b["betas"])
            assert a["weight_decay"] == b["weight_decay"] and a["eps"] == b["eps"]
            assert [gname[id(p)] for p in a["params"]] == b["params"], a["name"]      # same tensors, same order
    for mine in (od, od_f):
        a, b = mine.param_groups[0], gold["optimizer_D"][0]
        assert len(mine.param_groups) == len(gold["optimizer_D"]) == 1 and a["lr"] == b["lr"] and tuple(a["betas"]) == tuple(b["betas"])
        assert [dname[id(p)] for p in a["params"]] == b["params"]
    # every generator parameter is in exactly one group
    ids = [id(p) for g in og.param_groups for p in g["params"]]
    assert len(ids) == len(set(ids)) == len(list(G.parameters()))


def test_parameter_ema_matches_reference_ema(pkg, gold):
    ts = importlib.import_module("3dhumangan_b200.train_step")
    G, _, _ = rec.modules(pkg)
    params = list(G.parameters())
    a, counts = rec.ema_run(params, lambda ps: ts.ParameterEMA(ps, decay=rec.EMA_DECAY))
    assert counts == gold["ema_num_updates"]
    assert len(a.shadow_params) == gold["ema_shadow_count"]

    def check(tensors):
        sample, moments = rec.ema_summary(tensors)
        assert torch.allclose(sample, gold["ema_sample"], rtol=1e-6, atol=1e-8)
        assert torch.allclose(moments, gold["ema_moments"], rtol=1e-6, atol=1e-8)

    check(a.shadow_params)
    # copy_to writes the averages into the parameters that require grad, in order
    a.copy_to(G.parameters())
    check(list(G.parameters()))


@pytest.mark.parametrize("gan_lambda", [1.0, 0.0])
def test_r1_penalty_matches_phase_trainer(gan_lambda, gold):
    """`train_step.r1_penalty` against the reference's `_calculate_r1_regularization` (phase_trainer.py:259-294) on a small
    differentiable stand-in for the discriminator: value and the gradient the penalty sends into the parameters (the double
    backward), with an enabled-style scale factor going through `scaler.scale` / `get_scale`."""
    ts = importlib.import_module("3dhumangan_b200.train_step")
    ref = (float(gold[f"r1_{gan_lambda}_value"]), gold[f"r1_{gan_lambda}_grad_a"], gold[f"r1_{gan_lambda}_grad_b"])
    got = rec.r1_run(ts.r1_penalty, gan_lambda)
    assert got[0] == pytest.approx(ref[0], rel=1e-12, abs=1e-18)
    assert torch.allclose(got[1], ref[1], rtol=1e-10, atol=1e-16) and torch.allclose(got[2], ref[2], rtol=1e-10, atol=1e-16)
    if gan_lambda > 0:
        assert ref[0] > 0


# ----------------------------------------------------------------------------------------------------------------------
# the composition of the two steps: the reference's own `_train_discriminator` / `_train_generator` (phase_trainer.py:344-560),
# unmodified, against `train_step.Trainer.train_discriminator / train_generator` on the same stand-in networks
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("gan_lambda,do_r1", [(0.0, False), (0.0, True), (1.0, True)])
def test_step_composition_matches_phase_trainer(pkg, gan_lambda, do_r1, gold):
    ts = importlib.import_module("3dhumangan_b200.train_step")
    L, LD, meta, phase, images, labels, x, z_d, z_g = rec.composition_case(gan_lambda, do_r1)
    key = rec.composition_key(gan_lambda, do_r1)
    Gm, Dm = rec.StandInG(L), rec.StandInD(LD)
    dgrads = [gold[f"{key}_d_grad_{i}"] for i in range(len(list(Dm.parameters())))]
    ggrads = [gold[f"{key}_g_grad_{i}"] for i in range(len(list(Gm.parameters())))]
    t = ts.Trainer(Gm, Dm, meta, amp=False, ddp=False, fused=False)
    batch = dict(images=images, labels=labels, cond={"x": x}, z_d=z_d, z_g=z_g)
    d_mine = t.train_discriminator(batch)
    for p, r in zip(Dm.parameters(), dgrads):
        assert torch.allclose(p.grad, r, rtol=1e-5, atol=1e-7), float((p.grad - r).abs().max())
    assert float(d_mine) == pytest.approx(float(gold[key + "_d_loss"]), rel=1e-6)
    g_mine = t.train_generator(batch)
    for p, r in zip(Gm.parameters(), ggrads):
        assert torch.allclose(p.grad, r, rtol=1e-5, atol=1e-7), float((p.grad - r).abs().max())
    assert float(g_mine) == pytest.approx(float(gold[key + "_g_loss"]), rel=1e-6, abs=1e-12)
    # learning rate 0, no clipping: both steps ran their optimiser / EMA tail without moving a parameter
    for i, p in enumerate(list(Gm.parameters()) + list(Dm.parameters())):
        assert torch.equal(p.detach(), gold[f"{key}_param_{i}"])


@pytest.mark.parametrize("name", ["MAP3DBN", "MAP3DBN512", "MAP3DBN512L"])
def test_curricula_match_reference_configs(pkg, name, gold):
    """`3dhumangan_b200.configs` (the drop-in `configs` package) against the reference's `configs/map3d.py` + `extract_metadata`
    (configs/__init__.py) for every shipped curriculum at steps on both sides of every schedule boundary."""
    cur_m = getattr(pkg.configs, name)
    ref = gold["curricula"][name]
    for step, i in ref["steps"]:
        a = ref["metadata"][i]
        b = pkg.configs.extract_metadata(cur_m, step)
        for k, v in a.items():
            assert k in b, (name, step, k)
            if k == "neural_field_cls":
                assert v == (b[k] if isinstance(b[k], str) else b[k].__name__)
            else:
                assert b[k] == v, (name, step, k, v, b[k])
        extra = set(b) - set(a)
        assert all(k.startswith("hg_") for k in extra), (name, step, extra)


def test_trainer_refuses_the_branches_it_does_not_mirror():
    ts = importlib.import_module("3dhumangan_b200.train_step")
    meta = dict(latent_dim=5, label_dim=7, gan_lambda=0.0, segmentation_lambda=1.0, r1_lambda=0.0, grad_clip=1.0, gen_lr=0.0, disc_lr=0.0,
                betas=(0.0, 0.9), weight_decay=0, appearance_codes_lr_mul=1.0, mapping_net_lr_mul=1.0, neural_field_lr_mul=1.0,
                phases=[{"name": "uncond", "uncond": True, "rotate": True, "gen_modal": "rgbs_render", "do_r1": False}])
    t = ts.Trainer(rec.StandInG(5), rec.StandInD(7), meta, amp=False, ddp=False, fused=False)
    batch = dict(images=torch.zeros(2, 3, 8, 8), labels=torch.zeros(2, 8, 8, dtype=torch.long), cond={"x": torch.zeros(2, 6, 8, 8)})
    with pytest.raises(RuntimeError, match="not built"):
        t.train_discriminator(batch)
    with pytest.raises(RuntimeError, match="not built"):
        t.train_generator(batch)


def test_activation_table_matches_reference_bias_act(gold):
    """ops/bias_act.ACTIVATIONS (id, default alpha, default gain, which tensor the backward keeps, second derivative) against the
    reference's `activation_funcs` (lib/components/ops/bias_act.py:22-32) -- the ids are what the C ABI's `act` argument means."""
    mine = importlib.import_module("3dhumangan_b200.ops.bias_act").ACTIVATIONS
    cuda_acts = gold["activations"]
    assert set(mine) == set(cuda_acts)
    for k, (cuda_idx, def_alpha, def_gain, ref, has_2nd_grad) in cuda_acts.items():
        aid, alpha, gain, keep, second = mine[k]
        assert aid == cuda_idx and alpha == pytest.approx(def_alpha) and gain == pytest.approx(def_gain)
        assert keep == ref and second == has_2nd_grad


@pytest.mark.parametrize("tune,variant", rec.GET_CONFIG)
def test_get_config_matches_reference(pkg, tune, variant, gold):
    """`configs.get_config(opt)` (configs/__init__.py:49-76: curriculum lookup, neural-field class resolution, the two `--tune`
    sweeps) on a deep copy of the package's curriculum."""
    a = next(e for e in gold["get_config"] if e["tune"] == tune and e["variant"] == variant)
    mine = pkg.configs
    name = rec.GET_CONFIG_NAME
    saved_m = copy.deepcopy(getattr(mine, name))
    try:
        opt = types.SimpleNamespace(config=name, tune=tune, variant=variant)
        b = mine.get_config(opt)
        assert a["name"] == b["name"] and a["map3d_mode"] == b["map3d_mode"]
        assert a["neural_field_cls"] == b["neural_field_cls"].__name__
        for k, v in a["stages"]:
            assert v == b[k], (k, v, b[k])
    finally:
        setattr(mine, name, saved_m)
