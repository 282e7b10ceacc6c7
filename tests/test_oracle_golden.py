"""The oracle (CPU restatement) against the committed golden fixtures, which were produced by the UNMODIFIED
reference UNet3D (tests/golden/make_golden.py): training-mode forward, Dice and gradients, and the reference's state-dict
spec and eval-mode forward."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import UNetConfig, make_state_dict, unet3d_forward, unet3d_state_dict_spec, dice_loss

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
from recipe import CASES, REFERENCE_CASES, SUB2, golden_inputs, dropout_mask, reference_eval_input, stored_spec  # noqa: E402

FAST = ["c1_bw8_32", "bw16_n2_32", "bw8_convT_32", "c5like_1ch_5lev_32", "bw8_nonpow2_24x32x40"]


def _oracle_run(name, dtype=torch.float64):
    kw, shape = CASES[name]
    cfg = UNetConfig(**kw)
    sd = {k: v.requires_grad_(True) for k, v in make_state_dict(cfg, seed=0, dtype=dtype).items()}
    x, t, g3 = golden_inputs(shape, cfg.n_outputs)
    mask = dropout_mask(shape[0], cfg.enc_widths()[0], cfg.dropout, g3)
    logits = unet3d_forward(sd, x.to(dtype), cfg, dropout_mask=mask)
    loss = dice_loss(logits, t)
    loss.backward()
    with torch.no_grad():
        logits_eval = unet3d_forward(sd, x.to(dtype), cfg)
    return cfg, sd, logits.detach(), loss.detach(), logits_eval


@pytest.mark.parametrize("name", FAST)
def test_oracle_matches_golden(name, golden_dir):
    gold = np.load(os.path.join(golden_dir, name + ".npz"))
    cfg, sd, logits, loss, logits_eval = _oracle_run(name)
    sub = (slice(None), slice(None), slice(None, None, 4), slice(None, None, 4), slice(None, None, 4))
    np.testing.assert_allclose(logits[sub].numpy(), gold["logits_sub4"], rtol=0, atol=2e-6)
    np.testing.assert_allclose(logits_eval[sub].numpy(), gold["logits_eval_sub4"], rtol=0, atol=2e-6)
    assert abs(float(logits.norm()) - float(gold["logits_norm"])) <= 1e-9 * float(gold["logits_norm"])
    assert abs(float(loss) - float(gold["dice"])) < 1e-12
    keys = [str(k) for k in gold["grad_keys"]]
    norms = {k: float(n) for k, n in zip(keys, gold["grad_norms"])}
    assert sorted(sd) == keys
    for k, p in sd.items():
        assert abs(float(p.grad.norm()) - norms[k]) <= 1e-8 * max(norms[k], 1e-12), k
        gk = "grad::" + k
        if gk in gold:
            np.testing.assert_allclose(p.grad.numpy(), gold[gk], rtol=0, atol=1e-6 * max(1.0, float(np.abs(gold[gk]).max())))


def test_oracle_fp32_within_documented_noise(golden_dir):
    """fp32 CPU vs fp64: the noise floor the parity tolerance (1e-3) is quoted against (SURVEY 8c: 8.7e-7)."""
    gold = np.load(os.path.join(golden_dir, "c1_bw8_32.npz"))
    assert float(gold["fp32_vs_fp64_logits_rel"]) < 5e-6
    _, _, logits32, loss32, _ = _oracle_run("c1_bw8_32", torch.float32)
    _, _, logits64, loss64, _ = _oracle_run("c1_bw8_32", torch.float64)
    assert float((logits32.double() - logits64).norm() / logits64.norm()) < 5e-6
    assert abs(float(loss32) - float(loss64)) < 1e-6


def test_state_dict_spec_counts():
    spec = unet3d_state_dict_spec(UNetConfig(n_features=4, n_outputs=3, base_width=32))
    assert len(spec) == 90                                       # SURVEY appendix B
    n_params = sum(int(np.prod(s)) for _, s in spec)
    assert abs(n_params - 23.97e6) < 0.02e6                      # SURVEY 8a: 23.97 M (trilinear)
    spec_t = unet3d_state_dict_spec(UNetConfig(n_features=4, n_outputs=3, base_width=32, use_transposed_convolutions=True))
    assert abs(sum(int(np.prod(s)) for _, s in spec_t) - 25.35e6) < 0.02e6


@pytest.mark.parametrize("name", sorted(REFERENCE_CASES))
def test_oracle_matches_reference_fixture(name, golden_dir):
    gold = np.load(os.path.join(golden_dir, "reference_unet3d.npz"))
    kw, shape = REFERENCE_CASES[name]
    cfg = UNetConfig(**kw)
    assert stored_spec(gold, name) == unet3d_state_dict_spec(cfg)
    sd = make_state_dict(cfg, seed=3, dtype=torch.float64)
    with torch.no_grad():
        b = unet3d_forward(sd, reference_eval_input(shape), cfg)
    assert float(np.abs(b[SUB2].numpy() - gold["eval_sub2::" + name]).max()) < 1e-10
    assert abs(float(b.norm()) - float(gold["eval_norm::" + name])) <= 1e-12 * float(gold["eval_norm::" + name])
