"""Checkpoint boundary (CPU, no kernels): ``utils.load_model`` (utils/utils.py:294-360) and the
``Trainer.save_checkpoint`` dict layout (bin/train.py:112-186) round-trip through the mirror modules; a checkpoint
written by the REAL reference (rebuilt from tests/golden/checkpoint_ref.npz) loads into the mirror and checkpoints
written by the mirror have the layout the reference modules and optimizer load."""
import sys

import numpy as np
import torch
import yaml

from helpers import load_golden
from oracle import synth

HIFI_SMALL = dict(in_channels=80, out_channels=1, channels=64, kernel_size=7, upsample_scales=[8, 8, 2, 2],
                  upsample_kernel_sizes=[16, 16, 4, 4], resblock_kernel_sizes=[3, 7, 11],
                  resblock_dilations=[[1, 3, 5], [1, 3, 5], [1, 3, 5]])
MB_SMALL = dict(in_channels=80, out_channels=4, kernel_size=7, channels=96, upsample_scales=[2, 2, 2], stack_kernel_size=3, stacks=2)


def _fill(m, seed):
    sd = synth.synth_state_dict([(k, tuple(v.shape)) for k, v in m.state_dict().items()], seed, 1.0)
    m.load_state_dict(sd)
    return sd


def test_checkpoint_dict_round_trip(tmp_path):
    from parallelwavegan_b200 import models, optimizers, utils

    g, d = models.HiFiGANGenerator(**HIFI_SMALL), models.HiFiGANMultiScaleMultiPeriodDiscriminator()
    sdg, sdd = _fill(g, 1), _fill(d, 2)
    og, od = optimizers.RAdam(g.parameters(), lr=1e-4, eps=1e-6), optimizers.FusedAdam(d.parameters(), lr=2e-4, betas=(0.5, 0.9))
    for opt in (og, od):  # populate the state as a step would (the kernels themselves need a GPU)
        for p in opt.param_groups[0]["params"]:
            opt._init_state(p)
            opt.state[p]["exp_avg"].normal_()
            opt._bump(p)
    sg = torch.optim.lr_scheduler.StepLR(og, step_size=10, gamma=0.5)
    sdl = torch.optim.lr_scheduler.StepLR(od, step_size=10, gamma=0.5)
    path = str(tmp_path / "exp" / "checkpoint-7steps.pkl")
    utils.save_checkpoint(path, {"generator": g, "discriminator": d}, {"generator": og, "discriminator": od},
                          {"generator": sg, "discriminator": sdl}, steps=7, epochs=1)
    ck = torch.load(path, map_location="cpu")
    assert sorted(ck.keys()) == ["epochs", "model", "optimizer", "scheduler", "steps"]  # train.py:121-146
    assert sorted(ck["model"].keys()) == sorted(ck["optimizer"].keys()) == sorted(ck["scheduler"].keys()) == ["discriminator", "generator"]
    assert list(ck["model"]["generator"].keys()) == list(sdg.keys()) and list(ck["model"]["discriminator"].keys()) == list(sdd.keys())
    assert sorted(ck["optimizer"]["generator"]["state"][0].keys()) == ["exp_avg", "exp_avg_sq", "step"]
    g2, d2 = models.HiFiGANGenerator(**HIFI_SMALL), models.HiFiGANMultiScaleMultiPeriodDiscriminator()
    og2, od2 = optimizers.RAdam(g2.parameters(), lr=1.0), optimizers.FusedAdam(d2.parameters(), lr=1.0)
    steps, epochs = utils.load_checkpoint(path, {"generator": g2, "discriminator": d2}, {"generator": og2, "discriminator": od2})
    assert (steps, epochs) == (7, 1)
    for (k, a), (_, b) in zip(g.state_dict().items(), g2.state_dict().items()):
        assert torch.equal(a, b), k
    p0, q0 = next(iter(g.parameters())), next(iter(g2.parameters()))
    assert torch.equal(og.state[p0]["exp_avg"], og2.state[q0]["exp_avg"]) and og2.state[q0]["step"] == 1
    assert og2.param_groups[0]["lr"] == og.param_groups[0]["lr"]


def test_load_model_from_checkpoint_dir(tmp_path):
    """load_model: config.yml + stats.npy next to the checkpoint, typo-key workaround, PQMF attach with the
    version-gated defaults (utils.py:322-357)."""
    from parallelwavegan_b200 import layers, models, utils

    g = models.MelGANGenerator(**MB_SMALL)
    _fill(g, 3)
    d = tmp_path / "mb"
    d.mkdir()
    torch.save({"model": {"generator": g.state_dict()}}, str(d / "checkpoint-1steps.pkl"))
    cfg = {"generator_type": "MelGANGenerator", "generator_params": MB_SMALL, "format": "npy", "version": "0.4.0"}
    with open(d / "config.yml", "w") as f:
        yaml.dump(cfg, f)
    stats = np.stack([np.linspace(-1, 1, 80), np.linspace(0.5, 2, 80)]).astype(np.float32)
    np.save(str(d / "stats.npy"), stats)
    m = utils.load_model(str(d / "checkpoint-1steps.pkl"))
    assert isinstance(m, models.MelGANGenerator) and isinstance(m.pqmf, layers.PQMF) and m.pqmf.subbands == 4
    ref_old = layers.PQMF(4, taps=62, cutoff_ratio=0.15, beta=9.0)  # version <= 0.4.2 defaults
    assert torch.equal(m.pqmf.analysis_filter, ref_old.analysis_filter)
    assert torch.equal(m.mean, torch.from_numpy(stats[0])) and torch.equal(m.scale, torch.from_numpy(stats[1]))
    msd = m.state_dict()
    for k, a in g.state_dict().items():
        assert torch.equal(a, msd[k]), k
    cfg2 = dict(cfg, version="0.5.0")
    m2 = utils.load_model(str(d / "checkpoint-1steps.pkl"), config=cfg2)
    assert torch.equal(m2.pqmf.analysis_filter, layers.PQMF(4).analysis_filter)
    # typo key of old HiFi-GAN configs (utils.py:322-326)
    hp = {("upsample_kernal_sizes" if k == "upsample_kernel_sizes" else k): v for k, v in HIFI_SMALL.items()}
    h = models.HiFiGANGenerator(**HIFI_SMALL)
    _fill(h, 4)
    torch.save({"model": {"generator": h.state_dict()}}, str(d / "h.pkl"))
    mh = utils.load_model(str(d / "h.pkl"), config={"generator_type": "HiFiGANGenerator", "generator_params": hp, "format": "npy"}, stats=str(d / "stats.npy"))
    assert isinstance(mh, models.HiFiGANGenerator)


def _reference_checkpoint(meta, gold):
    """The checkpoint the real reference wrote (tests/golden/checkpoint_ref.npz, oracle/make_golden.py), rebuilt from
    its seeds: synthetic weights, one RAdam step (oracle.ref_optim.radam_step, the reference's own tensor ops) on
    seeded gradients; checked against the checksums and the first parameter's state the reference recorded."""
    from oracle import ref_optim

    g_sd = synth.synth_state_dict(meta["g_spec"], meta["g_seed"], meta["gain"])
    d_sd = synth.synth_state_dict(meta["d_spec"], meta["d_seed"], meta["gain"])
    (group,) = meta["g_param_groups"]
    assert len(group["params"]) == len(g_sd)  # every generator state-dict entry is a parameter, in parameter order
    state = {}
    for i, p in enumerate(g_sd.values()):
        m, v = torch.zeros_like(p), torch.zeros_like(p)
        grad = synth.randn(p.shape, meta["grad_seed"] + i, meta["grad_scale"])
        ref_optim.radam_step(p, grad, m, v, meta["step"], group["lr"], tuple(group["betas"]), group["eps"], group["weight_decay"])
        s = {"step": meta["step"], "exp_avg": m, "exp_avg_sq": v}
        state[i] = {k: s[k] for k in meta["state_keys"]}
    for sd, key in ((g_sd, "g_checksum"), (d_sd, "d_checksum"),
                    ({i: s["exp_avg"] for i, s in state.items()}, "exp_avg_checksum"),
                    ({i: s["exp_avg_sq"] for i, s in state.items()}, "exp_avg_sq_checksum")):
        assert abs(synth.checksum(sd) - meta[key]) <= 1e-12 * abs(meta[key]), key
    assert torch.equal(state[0]["exp_avg"], gold["exp_avg_p0"]) and torch.equal(state[0]["exp_avg_sq"], gold["exp_avg_sq_p0"])
    groups = {net: [dict(gr, betas=tuple(gr["betas"])) for gr in meta[f"{net[0]}_param_groups"]] for net in ("generator", "discriminator")}
    return {"model": {"generator": g_sd, "discriminator": d_sd},
            "optimizer": {"generator": {"state": state, "param_groups": groups["generator"]},
                          "discriminator": {"state": {}, "param_groups": groups["discriminator"]}},
            "scheduler": {"generator": {}, "discriminator": {}}, "steps": 1, "epochs": 0}


def test_checkpoints_interchange_with_the_real_reference(tmp_path):
    from parallelwavegan_b200 import models, optimizers, utils

    meta, gold = load_golden("checkpoint_ref")
    assert meta["g_kwargs"] == HIFI_SMALL

    # reference -> mirror
    ck_ref = _reference_checkpoint(meta, gold)
    path = str(tmp_path / "ref.pkl")
    torch.save(ck_ref, path)
    m = utils.load_model(path, config={"generator_type": "HiFiGANGenerator", "generator_params": HIFI_SMALL, "format": "npy"})
    for (k, a), (k2, b) in zip(ck_ref["model"]["generator"].items(), m.state_dict().items()):
        assert k == k2 and torch.equal(a, b)
    g2, d2 = models.HiFiGANGenerator(**HIFI_SMALL), models.HiFiGANMultiScaleMultiPeriodDiscriminator()
    o2 = optimizers.RAdam(g2.parameters(), lr=1.0)
    utils.load_checkpoint(path, {"generator": g2, "discriminator": d2}, {"generator": o2, "discriminator": optimizers.FusedAdam(d2.parameters())})
    p_new = next(iter(g2.parameters()))
    assert torch.equal(gold["exp_avg_p0"], o2.state[p_new]["exp_avg"]) and o2.state[p_new]["step"] == 1
    assert o2.param_groups[0]["lr"] == 1e-3
    # mirror -> reference: a strict load_state_dict into the reference modules needs the same names and shapes
    utils.save_checkpoint(str(tmp_path / "ours.pkl"), {"generator": g2, "discriminator": d2},
                          {"generator": o2, "discriminator": optimizers.FusedAdam(d2.parameters())})
    ck = torch.load(str(tmp_path / "ours.pkl"), map_location="cpu")
    for net in ("generator", "discriminator"):
        assert {k: list(v.shape) for k, v in ck["model"][net].items()} == {k: s for k, s in meta[f"{net[0]}_spec"]}, net
    # the reference RAdam inherits load_state_dict from torch.optim.Optimizer (radam.py) and its step() reads the
    # state keys it writes
    (group,) = meta["g_param_groups"]
    ro2 = torch.optim.Optimizer([torch.nn.Parameter(torch.zeros(s)) for _, s in meta["g_spec"]],
                                dict({k: v for k, v in group.items() if k != "params"}, lr=5.0))
    ro2.load_state_dict(ck["optimizer"]["generator"])
    assert ro2.param_groups[0]["lr"] == 1e-3
    assert all(sorted(s) == sorted(meta["state_keys"]) for s in ck["optimizer"]["generator"]["state"].values())
