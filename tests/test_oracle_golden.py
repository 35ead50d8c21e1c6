"""Pins oracle/vit3d_oracle.py (the CPU restatement) against golden vectors produced by
the unmodified reference (oracle/gen_golden.py).  CPU only."""
import os

import numpy as np
import pytest
import torch

from oracle import vit3d_oracle as O
from tests.helpers import CASES, assert_stats_close, assert_stats_equal, case_setup, load_golden, stats, unpack_masks

FAST = ["tiny", "shipped", "conf5", "conf18", "shipped_p8"]


def test_init_matches_reference_constructor_rng():
    g = load_golden("init_seed42")
    for name, (args, _) in CASES.items():
        cfg = O.get_config(*args)
        sd = O.init_state_dict(cfg, seed=42, randomize_tokens=False)
        keys = [k[len(name) + 1:] for k in g.files if k.startswith(name + "/")]
        assert sorted(keys) == sorted(sd.keys())
        for k in keys:
            assert_stats_equal(stats(sd[k]), g[f"{name}/{k}"], f"{name}/{k}")


@pytest.mark.parametrize("name", list(CASES))
def test_forward_matches_reference(name):
    g = load_golden(name)
    cfg, sd, x, y, w = case_setup(name)
    assert_stats_equal(stats(x), g["x_stats"], "x")
    for k, v in sd.items():
        assert_stats_equal(stats(v), g["sd_stats/" + k], k)
    logits, probs, enc = O.vit_forward(sd, cfg, x)
    np.testing.assert_allclose(logits.numpy(), g["logits"], atol=2e-5, rtol=0)
    np.testing.assert_allclose(enc[:, 0].numpy(), g["cls_feature"], atol=5e-5, rtol=0)
    assert_stats_close(stats(enc), g["enc_stats"], 1e-5, 1e-6, "enc")
    for i, p in enumerate(probs):
        assert_stats_close(stats(p), g[f"probs_stats/{i}"], 1e-5, 1e-6, f"probs{i}")
    xu = O.synth_volumes(x.shape[0], seed=43, kind="unit")
    np.testing.assert_allclose(O.vit_forward(sd, cfg, xu)[0].numpy(), g["logits_unit"], atol=2e-5, rtol=0)
    if name == "tiny":
        np.testing.assert_allclose(enc.numpy(), g["enc"], atol=2e-5)
        np.testing.assert_allclose(probs[0].numpy(), g["probs0"], atol=1e-6)


@pytest.mark.parametrize("name", FAST)
def test_loss_and_grads_eval_mode(name):
    g = load_golden(name)
    cfg, sd, x, y, w = case_setup(name)
    loss, grads, _ = O.vit_loss_and_grads(sd, cfg, x, y, w)
    assert abs(float(loss) - float(g["loss_eval"])) < 2e-6
    gscale = max(float(g["grad_eval_stats/" + k][1]) for k in grads)   # key.bias grads are exactly 0 in maths
    for k, gr in grads.items():
        assert_stats_close(stats(gr), g["grad_eval_stats/" + k], 2e-4, 1e-6 * gscale, k)
        if name == "tiny":
            np.testing.assert_allclose(gr.numpy(), g["grad_eval/" + k], rtol=2e-3,
                                       atol=1e-6 * max(1.0, float(np.abs(g["grad_eval/" + k]).max())))


@pytest.mark.parametrize("name", ["tiny", "conf5"])
def test_loss_and_grads_train_mode_with_reference_masks(name):
    """Dropout parity by mask injection: the masks the reference drew are replayed."""
    g = load_golden(name)
    cfg, sd, x, y, w = case_setup(name)
    masks = unpack_masks(g)
    assert len(masks) == 1 + 2 * cfg.transformer["num_layers"]
    loss, grads, _ = O.vit_loss_and_grads(sd, cfg, x, y, w, masks=masks)
    assert abs(float(loss) - float(g["loss_train"])) < 2e-6
    gscale = max(float(g["grad_train_stats/" + k][1]) for k in grads)
    for k, gr in grads.items():
        assert_stats_close(stats(gr), g["grad_train_stats/" + k], 2e-4, 1e-6 * gscale, k)


def test_ensemble_matches_reference():
    g = load_golden("ensemble_5_9_11")
    cfgs = [O.north_star_config(c) for c in (5, 9, 11)]
    members = []
    for j, c in enumerate(cfgs):
        members.append(O.init_state_dict(c, seed=42 + j))
    sd = O.ensemble_state_dict(members, seed=7)
    assert len(sd) == int(g["n_keys"])
    np.testing.assert_array_equal(sd["classifier.weight"].numpy(), g["classifier.weight"])
    x = O.synth_volumes(3, seed=42, kind="img")
    out = O.ensemble_forward(sd, cfgs, x)
    np.testing.assert_allclose(out.numpy(), g["out"], atol=2e-6)
    assert ((out > 0.5) == (torch.from_numpy(g["out"]) > 0.5)).all()


def test_north_star_table():
    # README.md:24-44 order: mlp {2048,3072} x L {4,6,8} x heads {4,8,16}
    c5, c9, c11, c18 = (O.north_star_config(c) for c in (5, 9, 11, 18))
    assert (c5.transformer.mlp_dim, c5.transformer.num_layers, c5.transformer.num_heads) == (2048, 6, 8)
    assert (c9.transformer.mlp_dim, c9.transformer.num_layers, c9.transformer.num_heads) == (2048, 8, 16)
    assert (c11.transformer.mlp_dim, c11.transformer.num_layers, c11.transformer.num_heads) == (3072, 4, 8)
    assert (c18.transformer.mlp_dim, c18.transformer.num_layers, c18.transformer.num_heads) == (3072, 8, 16)
    assert abs(O.fwd_flops_per_volume(c5) / 1e9 - 1.0903) < 1e-3
    assert abs(O.fwd_flops_per_volume(c18) / 1e9 - 1.9850) < 1e-3


def test_real_volume_fixture():
    g = load_golden("real_volumes")
    u8 = torch.from_numpy(g["u8"]).float().permute(0, 4, 1, 2, 3).contiguous()
    x = u8 - u8.mean()
    cfg = O.north_star_config(5)
    sd = O.init_state_dict(cfg, seed=42)
    logits = O.vit_forward(sd, cfg, x)[0]
    np.testing.assert_allclose(logits.numpy(), g["logits_conf5"], atol=3e-5)
